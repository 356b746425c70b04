"""Batched host API over the C ABI: the device-resident counterparts of the reference's
DynSAM / StaticSAM / DraftModel.lookup+update / eval_posterior+select_indices.

Everything here marshals torch tensors (device memory + the current stream) into
libsamd_b200.so calls; no arithmetic of the hot path runs in Python.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _cabi as K


def _i32(t: torch.Tensor) -> torch.Tensor:
    # device memory, or pinned host memory (mapped into the device address space under UVA: zero-copy I/O)
    assert t.dtype == torch.int32 and (t.is_cuda or t.is_pinned()) and t.is_contiguous(), \
        "expected a contiguous int32 CUDA (or pinned host) tensor"
    return t


class DynSamBatch:
    """`n_requests` independent dynamic suffix automata in HBM (samd/sam/dyn_sam.py:8-113)."""

    def __init__(self, n_requests: int, max_tokens: int, device: Optional[torch.device] = None):
        K.require_device()
        self.device = torch.device(device if device is not None else "cuda")
        self.n_requests = int(n_requests)
        self.max_tokens = int(max_tokens)
        self._h = K.vp()
        with torch.cuda.device(self.device):
            K.check(K.lib().samd_dyn_create(self.n_requests, self.max_tokens, C.byref(self._h)), "samd_dyn_create")

    @property
    def handle(self):
        return self._h

    @property
    def nbytes(self) -> int:
        return int(K.lib().samd_dyn_bytes(self._h))

    def reset(self, mask: Optional[torch.Tensor] = None):
        """DynSAM.reset for the masked requests (uint8 CUDA tensor; None = all)."""
        if mask is not None:
            assert mask.dtype == torch.uint8 and mask.is_cuda and mask.numel() == self.n_requests
        with torch.cuda.device(self.device):
            K.check(K.lib().samd_dyn_reset(self._h, K.ptr(mask), K.stream_ptr()), "samd_dyn_reset")

    def export(self, request: int, with_text: bool = True):
        """Host copy of one request's automaton (synchronises) - for parity tests."""
        meta = np.zeros(8, dtype=np.int32)
        cap = 2 * self.max_tokens + 2
        link = np.zeros(cap, dtype=np.int32)
        length = np.zeros(cap, dtype=np.int32)
        endpos = np.zeros(cap, dtype=np.int32)
        text = np.zeros(cap, dtype=np.int32)
        as_p = lambda a: a.ctypes.data_as(K.c_i32p)
        with torch.cuda.device(self.device):
            K.check(K.lib().samd_dyn_export(self._h, int(request), as_p(meta), as_p(link), as_p(length), as_p(endpos),
                                            as_p(text) if with_text else None, cap), "samd_dyn_export")
        ns, n = int(meta[0]), int(meta[2])
        return dict(n_states=ns, last=int(meta[1]), max_length=n, cur_index=int(meta[3]), cur_length=int(meta[4]),
                    n_edges=int(meta[5]), overflow=int(meta[6]), n_clones=int(meta[7]), link=link[:ns], length=length[:ns],
                    min_endpos=endpos[:ns], text=text[:n + 1])

    def export_edges(self, request: int) -> np.ndarray:
        """[n_edges, 3] (state, token, target) of one request, per state in insertion order (synchronises)."""
        n_edges = int(self.meta()[request, 5])
        out = np.zeros((max(n_edges, 1), 3), dtype=np.int32)
        with torch.cuda.device(self.device):
            K.check(K.lib().samd_dyn_export_edges(self._h, int(request), out.ctypes.data_as(K.c_i32p), n_edges), "samd_dyn_export_edges")
        return out[:n_edges]

    def meta(self) -> np.ndarray:
        """[n_requests, 16] meta words of every request (synchronises): n_states, last, max_length, cur_index, cur_length,
        n_edges, overflow flags (1 = arena full, 2 = negative token), n_clones, link hops, lookup probes, last_link, ...,
        [14] = the longest cursor fallback chain seen."""
        m = np.zeros((self.n_requests, 16), dtype=np.int32)
        with torch.cuda.device(self.device):
            K.check(K.lib().samd_dyn_meta(self._h, m.ctypes.data_as(K.c_i32p)), "samd_dyn_meta")
        return m

    def check(self):
        """Raise when a request was handed a token it could not take (synchronises): a full arena (grow with grown())
        or a negative token id.  The step kernel only raises per-request flags - it never stops a launch - so callers
        that size `max_tokens` from prompt + max_new_tokens call this once at the end; DraftEngine.step documents it."""
        st = self.stats()
        if st["overflowed"]:
            raise K.SamdError(f"{st['overflowed']} request(s) ran out of arena capacity (max_tokens={self.max_tokens}): "
                              "tokens were not appended; grow the batch (DynSamBatch.grown) or size it for prompt + new tokens")
        if st["bad_tokens"]:
            raise K.SamdError(f"{st['bad_tokens']} request(s) were handed a negative token id (-1 marks a free edge slot)")

    def grown(self, new_max_tokens: int) -> "DynSamBatch":
        """A new batch with a larger capacity holding the same automata (samd_dyn_grow)."""
        new = DynSamBatch.__new__(DynSamBatch)
        new.device, new.n_requests, new.max_tokens = self.device, self.n_requests, int(new_max_tokens)
        new._h = K.vp()
        with torch.cuda.device(self.device):
            K.check(K.lib().samd_dyn_grow(self._h, int(new_max_tokens), C.byref(new._h)), "samd_dyn_grow")
        return new

    def copy_from(self, other: "DynSamBatch"):
        """Snapshot / restore of all arenas (device-to-device, stream ordered)."""
        with torch.cuda.device(self.device):
            K.check(K.lib().samd_dyn_copy(self._h, other.handle, K.stream_ptr()), "samd_dyn_copy")

    def stats(self) -> dict:
        out = np.zeros(8, dtype=np.int64)
        with torch.cuda.device(self.device):
            K.check(K.lib().samd_dyn_stats(self._h, out.ctypes.data_as(K.c_i64p)), "samd_dyn_stats")
        keys = ("n_states", "tokens", "n_edges", "n_clones", "extend_probes", "lookup_probes", "overflowed", "bad_tokens")
        return {k: int(v) for k, v in zip(keys, out)}

    def close(self):
        if self._h:
            K.lib().samd_dyn_destroy(self._h)
            self._h = K.vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class StaticSamDevice:
    """Read-only static suffix automaton in HBM (samd/sam/static_sam.py, samd_sam_only/sam/static_sam.py)."""

    def __init__(self, handle, device):
        self._h = handle
        self.device = device
        info = np.zeros(8, dtype=np.int64)
        K.check(K.lib().samd_static_info(self._h, info.ctypes.data_as(K.c_i64p)), "samd_static_info")
        self.n_states, self.n_edges, self.n_tokens, self.n_slots, self.nbytes, wc, self.n_clones, _ = (int(x) for x in info)
        self.with_counts = bool(wc)

    @property
    def handle(self):
        return self._h

    @staticmethod
    def build(docs: Sequence[Sequence[int]], eos: int, with_counts: bool = False,
              device: Optional[torch.device] = None, host_only: bool = False) -> "StaticSamDevice":
        """StaticSAM.build (static_sam.py:38-46): host construction, flat upload."""
        lens = np.fromiter((len(d) for d in docs), dtype=np.int64, count=len(docs))
        offs = np.zeros(len(docs) + 1, dtype=np.int64)
        np.cumsum(lens, out=offs[1:])
        flat = np.empty(int(offs[-1]), dtype=np.int32)
        for i, d in enumerate(docs):
            flat[offs[i]:offs[i + 1]] = d
        return StaticSamDevice.build_flat(flat, offs, eos, with_counts, device, host_only)

    @staticmethod
    def build_flat(flat: np.ndarray, offs: np.ndarray, eos: int, with_counts: bool = False,
                   device: Optional[torch.device] = None, host_only: bool = False) -> "StaticSamDevice":
        """host_only=True stops after the host construction (no CUDA device needed): the result
        can be exported / saved but not queried until upload()."""
        flat = np.ascontiguousarray(flat, dtype=np.int32)
        offs = np.ascontiguousarray(offs, dtype=np.int64)
        h = K.vp()
        args = (flat.ctypes.data_as(K.c_i32p), offs.ctypes.data_as(K.c_i64p), len(offs) - 1, int(eos), int(with_counts),
                C.byref(h))
        if host_only:
            K.check(K.lib().samd_static_build_host(*args), "samd_static_build_host")
            return StaticSamDevice(h, None)
        K.require_device()
        device = torch.device(device if device is not None else "cuda")
        with torch.cuda.device(device):
            K.check(K.lib().samd_static_build(*args), "samd_static_build")
        return StaticSamDevice(h, device)

    def upload(self, device: Optional[torch.device] = None):
        K.require_device()
        self.device = torch.device(device if device is not None else "cuda")
        with torch.cuda.device(self.device):
            K.check(K.lib().samd_static_upload(self._h), "samd_static_upload")
        return self

    def drop_host(self):
        """Free the host mirrors (export / save stop working, queries do not): 15 GB for a 125 M-token shard."""
        K.check(K.lib().samd_static_drop_host(self._h), "samd_static_drop_host")
        return self

    @staticmethod
    def load(path: str, device: Optional[torch.device] = None, host_only: bool = False) -> "StaticSamDevice":
        h = K.vp()
        if host_only:
            K.check(K.lib().samd_static_load_host(path.encode(), C.byref(h)), "samd_static_load_host")
            return StaticSamDevice(h, None)
        K.require_device()
        device = torch.device(device if device is not None else "cuda")
        with torch.cuda.device(device):
            K.check(K.lib().samd_static_load(path.encode(), C.byref(h)), "samd_static_load")
        return StaticSamDevice(h, device)

    def save(self, path: str):
        K.check(K.lib().samd_static_save(self._h, path.encode()), "samd_static_save")

    def export(self):
        n = self.n_states
        link = np.zeros(n, dtype=np.int32)
        length = np.zeros(n, dtype=np.int32)
        endpos = np.zeros(n, dtype=np.int32)
        as_p = lambda a: a.ctypes.data_as(K.c_i32p)
        count = topk = None
        if self.with_counts:
            count = np.zeros(n, dtype=np.int32)
            topk = np.zeros((n, 8, 2), dtype=np.int32)
        K.check(K.lib().samd_static_export(self._h, as_p(link), as_p(length), as_p(endpos),
                                           as_p(count) if count is not None else None,
                                           as_p(topk) if topk is not None else None), "samd_static_export")
        return dict(link=link, length=length, min_endpos=endpos, cnt_endpos=count, topk=topk)

    def set_l2_window(self, nbytes: int):
        with torch.cuda.device(self.device):
            K.check(K.lib().samd_static_set_l2_window(self._h, K.stream_ptr(), int(nbytes)), "samd_static_set_l2_window")

    def new_cursors(self, n_requests: int) -> torch.Tensor:
        """StaticSAM.reset (static_sam.py:28-30) for n_requests queries: (index, length) = (0, 0)."""
        return torch.zeros(n_requests, 2, dtype=torch.int32, device=self.device)

    def close(self):
        if self._h:
            K.lib().samd_static_destroy(self._h)
            self._h = K.vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class DraftEngine:
    """DraftModel.update + DraftModel.lookup for a batch of requests (samd/draft.py:52-79,
    samd_sam_only/draft.py:49-67): one `samd_step` launch per call, outputs stay on the device."""

    def __init__(self, dyn: DynSamBatch, static: Optional[StaticSamDevice] = None, flavour: int = K.FLAVOUR_SAMD,
                 n_predicts: int = 40, len_bias: int = 5, len_threshold: int = 5, alpha: float = 4.0):
        self.dyn, self.static = dyn, static
        self.flavour, self.n_predicts, self.len_bias, self.len_threshold, self.alpha = \
            int(flavour), int(n_predicts), int(len_bias), int(len_threshold), float(alpha)
        B, dev = dyn.n_requests, dyn.device
        self.static_cursor = static.new_cursors(B) if static is not None else None
        # every output is a view of ONE device buffer, so a host caller needs a single D2H copy:
        # [type | match_dyn | match_static | index_dyn | index_static | draft_len | draft (B x n_predicts)]
        n = self.n_predicts
        self.out_buf = torch.zeros(B * (6 + n), dtype=torch.int32, device=dev)
        f = lambda i: self.out_buf[i * B:(i + 1) * B]
        self.out_type, self.match_dyn, self.match_static = f(0), f(1), f(2)
        self.index_dyn, self.index_static, self.draft_len = f(3), f(4), f(5)
        self.draft = self.out_buf[6 * B:].view(B, n)
        self._args = K.StepArgs()
        self._io = None

    def reset(self, mask: Optional[torch.Tensor] = None):
        """DraftModel.reset (draft.py:47-50)."""
        self.dyn.reset(mask)
        if self.static_cursor is not None:
            if mask is None:
                self.static_cursor.zero_()
            else:
                self.static_cursor.masked_fill_(mask.bool().unsqueeze(1), 0)

    def step(self, tokens: Optional[torch.Tensor] = None, counts: Optional[torch.Tensor] = None,
             start_tok: Optional[torch.Tensor] = None, out_buf: Optional[torch.Tensor] = None):
        """update(tokens[:, :counts]) then lookup(start_tok); either half may be omitted.  `out_buf` (same
        layout as self.out_buf, device or pinned host memory) redirects every output.
        Token ids must be non-negative (-1 is the layout's free-slot marker) and a request's history must fit
        `dyn.max_tokens`: a violation never stops the launch, it raises the request's flag - `dyn.check()` reports it."""
        a = self._args
        a.dyn = self.dyn.handle
        a.stat = self.static.handle if self.static is not None else None
        a.static_cursor_dev = K.ptr(self.static_cursor)
        if tokens is not None:
            _i32(tokens)
            assert tokens.dim() == 2 and tokens.shape[0] == self.dyn.n_requests
            a.tokens_dev, a.token_stride = tokens.data_ptr(), tokens.shape[1]
            a.counts_dev = K.ptr(_i32(counts)) if counts is not None else None
        else:
            a.tokens_dev, a.token_stride, a.counts_dev = None, 0, None
        a.start_tok_dev = K.ptr(_i32(start_tok)) if start_tok is not None else None
        a.flavour, a.n_predicts, a.len_bias, a.len_threshold, a.alpha = \
            self.flavour, self.n_predicts, self.len_bias, self.len_threshold, self.alpha
        ob = self.out_buf if out_buf is None else _i32(out_buf)
        assert ob.numel() == self.out_buf.numel()
        base, B4 = ob.data_ptr(), 4 * self.dyn.n_requests
        a.out_type_dev, a.out_match_dyn_dev, a.out_match_static_dev = base, base + B4, base + 2 * B4
        a.out_index_dyn_dev, a.out_index_static_dev, a.out_draft_len_dev = base + 3 * B4, base + 4 * B4, base + 5 * B4
        a.out_draft_dev, a.draft_stride = base + 6 * B4, self.n_predicts
        with torch.cuda.device(self.dyn.device):
            K.check(K.lib().samd_step(C.byref(a), K.stream_ptr()), "samd_step")

    # ---- batch-1 host-facing calls (the drop-in DraftModel.update / lookup): argument blocks built once --------------
    def _fill_common(self, a):
        a.dyn = self.dyn.handle
        a.stat = self.static.handle if self.static is not None else None
        a.static_cursor_dev = K.ptr(self.static_cursor)
        a.flavour, a.n_predicts, a.len_bias, a.len_threshold, a.alpha = \
            self.flavour, self.n_predicts, self.len_bias, self.len_threshold, self.alpha

    def _make_current(self):
        """The arenas' device must be the current one for the launch; switching costs ~100 us, checking costs nothing."""
        idx = self.dyn.device.index
        if idx is not None and torch.cuda.current_device() != idx:
            torch.cuda.set_device(idx)

    def quick_update(self, tokens: torch.Tensor):
        """update(tokens [1, k] int32 on the device) with a pre-built argument block: a Python call costs the ctypes
        launch and nothing else (no tensor checks, no device context switch when the device is already current)."""
        a = self.__dict__.get("_qu_args")
        if a is None:
            a = self._qu_args = K.StepArgs()
            a.counts_dev = a.start_tok_dev = None
            a.out_type_dev = a.out_match_dyn_dev = a.out_match_static_dev = a.out_index_dyn_dev = None
            a.out_index_static_dev = a.out_draft_dev = a.out_draft_len_dev = None
            a.draft_stride = 0
        self._fill_common(a)
        a.tokens_dev, a.token_stride = tokens.data_ptr(), tokens.shape[-1]
        self._make_current()
        K.check(K.lib().samd_step(C.byref(a), torch.cuda.current_stream().cuda_stream), "samd_step")

    def host_lookup(self, start_token: int) -> np.ndarray:
        """lookup(start_token) for ONE request with the start token read from, and every output written to, mapped
        pinned host memory by the one launch; returns the output block as a numpy view (layout of `out_buf`) after one
        stream synchronise.  No fill / cat / copy kernels, no per-call tensor checks."""
        h = self.__dict__.get("_hl")
        if h is None:
            assert self.dyn.n_requests == 1
            start = torch.zeros(1, dtype=torch.int32).pin_memory()
            out = torch.zeros(self.out_buf.numel(), dtype=torch.int32).pin_memory()
            a = K.StepArgs()
            a.tokens_dev, a.token_stride, a.counts_dev = None, 0, None
            a.start_tok_dev = start.data_ptr()
            base = out.data_ptr()
            a.out_type_dev, a.out_match_dyn_dev, a.out_match_static_dev = base, base + 4, base + 8
            a.out_index_dyn_dev, a.out_index_static_dev, a.out_draft_len_dev = base + 12, base + 16, base + 20
            a.out_draft_dev, a.draft_stride = base + 24, self.n_predicts
            h = self._hl = (a, start, out, start.numpy(), out.numpy())
        a, start, out, start_np, out_np = h
        self._fill_common(a)
        start_np[0] = int(start_token)
        self._make_current()
        st = torch.cuda.current_stream()
        K.check(K.lib().samd_step(C.byref(a), st.cuda_stream), "samd_step")
        st.synchronize()
        return out_np

    # ---- host-buffer path: one H2D copy in, one launch, one D2H copy out ---------------------------
    def host_buffers(self, max_tokens_per_step: int = 8):
        """Pinned host staging buffers for step_host(): `inp` = [counts (B) | start (B) | tokens (B x k)],
        `out` = the layout of `out_buf`.  Returns (inp, out) int32 tensors."""
        B, k = self.dyn.n_requests, int(max_tokens_per_step)
        inp = torch.zeros(B * (2 + k), dtype=torch.int32).pin_memory()
        out = torch.zeros(self.out_buf.numel(), dtype=torch.int32).pin_memory()
        dev_in = torch.zeros(B * (2 + k), dtype=torch.int32, device=self.dyn.device)
        self._io = (dev_in, k)
        return inp, out

    HOST_MODE = "stage_in"      # measured best on B200 at 1024 requests (35.8 us host to host; zero_copy 39.8, stage_both 38.6, copy_engine 49.7)

    def step_host(self, inp: torch.Tensor, out: torch.Tensor, sync: bool = True, zero_copy: bool = True, mode: Optional[str] = None):
        """DraftModel.update + lookup with HOST inputs / outputs (pinned buffers from host_buffers()).  `mode`:
        "zero_copy"   the step kernel reads `inp` and writes `out` directly over PCIe (pinned memory is mapped into the
                      device address space) - one launch, no copies;
        "stage_in"    one staging-copy KERNEL (samd_stage_copy: 16-byte coalesced reads of `inp` into a device block),
                      then the step kernel on device inputs, writing `out` directly;
        "stage_both"  the same, and the outputs go to the device block first and leave through a second copy kernel;
        "copy_engine" H2D memcpy, the kernel, D2H memcpy (zero_copy=False selects this).
        Either way the work is captured once per (inp, out) pair and replayed as one graph launch.  By default waits
        until `out` is complete.  Measured host to host at 1024 requests: see DESIGN.md section 5."""
        if mode is None:
            mode = self.HOST_MODE if zero_copy else "copy_engine"
        # same buffers and settings as the last call: replay at once (the check below costs a few microseconds)
        quick = (self.n_predicts, self.len_bias, self.len_threshold, self.alpha, mode)
        last = self.__dict__.get("_host_quick")
        if last is not None and inp is last[0] and out is last[1] and quick == last[2]:
            self._host_graph.replay()
            if sync:
                torch.cuda.current_stream(self.dyn.device).synchronize()
            return
        if not (inp.is_pinned() and out.is_pinned()):
            raise K.SamdError("step_host needs pinned host buffers (DraftEngine.host_buffers())")
        if mode not in ("zero_copy", "stage_in", "stage_both", "copy_engine"):
            raise K.SamdError(f"step_host: unknown mode {mode!r}")
        if not hasattr(self, "_io"):
            raise K.SamdError("step_host before host_buffers()")
        dev_in, k = self._io
        B = self.dyn.n_requests
        if inp.numel() != dev_in.numel() or out.numel() != self.out_buf.numel():
            raise K.SamdError("step_host: buffers do not have the layout of host_buffers()")
        key = (inp.data_ptr(), out.data_ptr(), self.dyn.handle.value, self.flavour, self.n_predicts, self.len_bias,
               self.len_threshold, self.alpha, mode)
        if getattr(self, "_host_graph_key", None) != key:
            def stage(dst, src):
                K.check(K.lib().samd_stage_copy(dst.data_ptr(), src.data_ptr(), dst.numel() * 4, K.stream_ptr()), "samd_stage_copy")

            def work():
                if mode == "zero_copy":
                    self.step(inp[2 * B:].view(B, k), inp[:B], inp[B:2 * B], out_buf=out)
                elif mode == "copy_engine":
                    dev_in.copy_(inp, non_blocking=True)
                    self.step(dev_in[2 * B:].view(B, k), dev_in[:B], dev_in[B:2 * B])
                    out.copy_(self.out_buf, non_blocking=True)
                else:
                    stage(dev_in, inp)
                    if mode == "stage_in":
                        self.step(dev_in[2 * B:].view(B, k), dev_in[:B], dev_in[B:2 * B], out_buf=out)
                    else:
                        self.step(dev_in[2 * B:].view(B, k), dev_in[:B], dev_in[B:2 * B])
                        stage(out, self.out_buf)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.device(self.dyn.device), torch.cuda.graph(g):
                work()
            self._host_graph, self._host_graph_key = g, key
        self._host_quick = (inp, out, quick)
        self._host_graph.replay()
        if sync:
            torch.cuda.current_stream(self.dyn.device).synchronize()

    def tree_draft(self, start_tok: torch.Tensor, K_top: int = 8, max_paths: Optional[int] = None):
        """sam_only static tree for requests whose out_type is DRAFT_STATIC_TREE (after step())."""
        assert self.static is not None and self.static.with_counts
        B, dev, n = self.dyn.n_requests, self.dyn.device, self.n_predicts
        max_paths = max_paths or n
        if not hasattr(self, "tree_tokens"):
            mk = lambda *s: torch.zeros(*s, dtype=torch.int32, device=dev)
            self.tree_tokens, self.tree_parents, self.tree_depth = mk(B, n), mk(B, n), mk(B, n)
            self.tree_n, self.tree_shape = mk(B), mk(B, 2)
            self.tree_retrieve = mk(B, max_paths, n)
        with torch.cuda.device(dev):
            K.check(K.lib().samd_static_tree_draft(
                self.static.handle, B, self.out_type.data_ptr(), self.index_static.data_ptr(), self.match_static.data_ptr(),
                _i32(start_tok).data_ptr(), n, self.alpha, int(K_top), self.len_bias, self.tree_tokens.data_ptr(),
                self.tree_parents.data_ptr(), self.tree_depth.data_ptr(), self.tree_n.data_ptr(),
                self.tree_retrieve.data_ptr(), self.tree_retrieve.shape[1], self.tree_retrieve.shape[2],
                self.tree_shape.data_ptr(), K.stream_ptr()), "samd_static_tree_draft")

    _MASK_DTYPES = {torch.bfloat16: K.DTYPE_BF16, torch.float16: K.DTYPE_FP16, torch.float32: K.DTYPE_FP32}

    def assemble(self, cache_len: torch.Tensor, tokens: torch.Tensor, position_ids: torch.Tensor, n_nodes: torch.Tensor,
                 n_paths: torch.Tensor, retrieve: torch.Tensor, mask: torch.Tensor, done: Optional[torch.Tensor] = None):
        """samd_draft_assemble: the last step()'s sequence drafts and, for the requests typed DRAFT_STATIC_TREE, the last
        tree_draft()'s trees, as uniform batch buffers written into the caller's tensors (persistent ones when the call
        is captured in a graph): tokens [B, T] int32, position_ids [B, T] int64, n_nodes / n_paths [B] int32, retrieve
        [B, P, D] int32 and the additive mask [B, T, kv_len] in the LM dtype.  `done` [B] bool / uint8: finished
        requests get a one-node draft with no path (no KV row moves in the verify launch)."""
        B = self.dyn.n_requests
        T, kv_len = tokens.shape[1], mask.shape[2]
        for t in (tokens, n_nodes, n_paths, retrieve, cache_len):
            _i32(t)
        assert tokens.shape == (B, T) and position_ids.shape == (B, T) and position_ids.dtype == torch.int64
        assert position_ids.is_contiguous() and n_nodes.numel() == B and n_paths.numel() == B and cache_len.numel() == B
        assert retrieve.dim() == 3 and retrieve.shape[0] == B and mask.dim() == 3 and mask.shape[:2] == (B, T)
        assert mask.is_cuda and mask.is_contiguous()
        dt = self._MASK_DTYPES.get(mask.dtype)
        if dt is None:
            raise K.SamdError(f"unsupported mask dtype {mask.dtype} (bf16 / fp16 / fp32)")
        if done is not None:
            assert done.dtype in (torch.bool, torch.uint8) and done.is_cuda and done.is_contiguous() and done.numel() == B
        a = K.AssembleArgs()
        a.batch, a.n_nodes, a.n_paths, a.depth = B, T, retrieve.shape[1], retrieve.shape[2]
        a.type_dev, a.draft_dev, a.draft_stride = self.out_type.data_ptr(), self.draft.data_ptr(), self.n_predicts
        a.draft_len_dev = self.draft_len.data_ptr()
        if hasattr(self, "tree_tokens"):
            a.tree_tokens_dev, a.tree_parents_dev = self.tree_tokens.data_ptr(), self.tree_parents.data_ptr()
            a.tree_depth_dev, a.tree_stride, a.tree_n_dev = self.tree_depth.data_ptr(), self.n_predicts, self.tree_n.data_ptr()
            a.tree_retrieve_dev, a.tree_shape_dev = self.tree_retrieve.data_ptr(), self.tree_shape.data_ptr()
            a.tree_max_paths, a.tree_max_depth = self.tree_retrieve.shape[1], self.tree_retrieve.shape[2]
        a.cache_len_dev, a.done_dev, a.mask_dtype, a.kv_len = cache_len.data_ptr(), K.ptr(done), dt, kv_len
        a.out_tokens_dev, a.out_position_ids_dev = tokens.data_ptr(), position_ids.data_ptr()
        a.out_n_nodes_dev, a.out_n_paths_dev = n_nodes.data_ptr(), n_paths.data_ptr()
        a.out_retrieve_dev, a.out_mask_dev = retrieve.data_ptr(), mask.data_ptr()
        with torch.cuda.device(self.dyn.device):
            K.check(K.lib().samd_draft_assemble(C.byref(a), K.stream_ptr()), "samd_draft_assemble")


class Verifier:
    """Fused greedy verification + KV compaction (samd/utils.py:127-141, samd/samd_model.py:159-211,
    samd/cache.py:118-133) for a batch of requests: one persistent launch."""

    def __init__(self, max_batch: int, max_nodes: int, device: Optional[torch.device] = None):
        K.require_device()
        self.device = torch.device(device if device is not None else "cuda")
        self._h = K.vp()
        with torch.cuda.device(self.device):
            K.check(K.lib().samd_verify_create(int(max_batch), int(max_nodes), C.byref(self._h)), "samd_verify_create")
        self._args = K.VerifyArgs()
        self._kv_key = None
        self._kv_ptrs = None
        self._last_key, self._last_out = None, None

    def bind_kv(self, kv_tensors: Optional[List[torch.Tensor]]):
        """Register the 2L cache tensors [B, H, max_len, Dh] (key_cache + value_cache order)."""
        if kv_tensors is None:
            self._kv_key, self._kv_ptrs, self._kv_meta = None, None, None
            return
        key = tuple(t.data_ptr() for t in kv_tensors)
        if key == self._kv_key:
            return
        t0 = kv_tensors[0]
        assert t0.dim() == 4 and t0.stride(3) == 1
        es = t0.element_size()
        for t in kv_tensors:
            assert t.shape == t0.shape and t.stride() == t0.stride() and t.dtype == t0.dtype and t.device == t0.device
        self._kv_ptrs = torch.tensor(list(key), dtype=torch.int64, device=self.device)
        self._kv_meta = dict(n_kv=len(kv_tensors), n_heads=t0.shape[1], row_bytes=t0.shape[3] * es,
                             batch_stride=t0.stride(0) * es, head_stride=t0.stride(1) * es, pos_stride=t0.stride(2) * es)
        self._kv_key = key

    def verify(self, logits: torch.Tensor, tree_tokens: torch.Tensor, retrieve: Optional[torch.Tensor],
               cache_len: Optional[torch.Tensor] = None, move_kv: bool = True, n_nodes: Optional[torch.Tensor] = None,
               n_paths: Optional[torch.Tensor] = None, out: Optional[dict] = None, want_argmax: bool = False,
               want_topk: bool = False, recycle: Optional["RecycleTable"] = None) -> dict:
        """`want_topk`: also return out["topk"] [B, T, 8], the 8 largest logits of every row as indices (value
        descending, index ascending).  `recycle`: additionally update that Token-Recycle table in the same launch
        (TokenRecycle.update, token_recycle.py:39-47)."""
        want_topk = want_topk or recycle is not None
        if recycle is not None:
            recycle.ensure(logits.shape[-1], logits.device)
        # fast path: identical buffers as the previous call -> relaunch with the argument block as it is
        key = (logits.data_ptr(), logits.shape, logits.stride(), logits.dtype, tree_tokens.data_ptr(),
               None if retrieve is None else (retrieve.data_ptr(), retrieve.shape), K.ptr(cache_len), bool(move_kv),
               K.ptr(n_nodes), K.ptr(n_paths), None if out is None else out["tokens"].data_ptr(), want_argmax, self._kv_key,
               want_topk, None if recycle is None else recycle.table.data_ptr())
        if key == getattr(self, "_last_key", None) and out is self._last_out:
            with torch.cuda.device(self.device):
                K.check(K.lib().samd_verify_compact(self._h, C.byref(self._args), K.stream_ptr()), "samd_verify_compact")
            return out
        assert logits.is_cuda and logits.dim() == 3 and logits.stride(2) == 1
        B, T, V = logits.shape
        dt = {torch.bfloat16: K.DTYPE_BF16, torch.float16: K.DTYPE_FP16, torch.float32: K.DTYPE_FP32}.get(logits.dtype)
        if dt is None:
            raise K.SamdError(f"unsupported logits dtype {logits.dtype} (bf16 / fp16 / fp32)")
        _i32(tree_tokens)
        assert tree_tokens.shape == (B, T)
        a = self._args
        a.logits_dev, a.dtype, a.batch, a.n_nodes, a.vocab = logits.data_ptr(), dt, B, T, V
        a.batch_stride, a.row_stride = logits.stride(0), logits.stride(1)
        a.tree_tokens_dev = tree_tokens.data_ptr()
        a.n_nodes_dev = K.ptr(_i32(n_nodes)) if n_nodes is not None else None
        if retrieve is not None:
            _i32(retrieve)
            if retrieve.dim() == 2:
                a.n_paths, a.depth, a.retrieve_batch_stride = retrieve.shape[0], retrieve.shape[1], 0
            else:
                assert retrieve.shape[0] == B
                a.n_paths, a.depth, a.retrieve_batch_stride = retrieve.shape[1], retrieve.shape[2], retrieve.stride(0)
            a.retrieve_dev = retrieve.data_ptr()
            width = a.depth
        else:
            a.retrieve_dev, a.n_paths, a.depth, a.retrieve_batch_stride = None, 1, T, 0
            width = T
        a.n_paths_dev = K.ptr(_i32(n_paths)) if n_paths is not None else None
        if self._kv_ptrs is not None and move_kv and retrieve is not None:
            m = self._kv_meta
            a.kv_ptrs_dev, a.n_kv, a.n_heads, a.row_bytes = self._kv_ptrs.data_ptr(), m["n_kv"], m["n_heads"], m["row_bytes"]
            a.kv_batch_stride, a.kv_head_stride, a.kv_pos_stride = m["batch_stride"], m["head_stride"], m["pos_stride"]
            a.move_kv = 1
        else:
            a.kv_ptrs_dev, a.n_kv, a.move_kv = None, 0, 0
        a.cache_len_dev = K.ptr(_i32(cache_len)) if cache_len is not None else None
        fresh = out is None or out["tokens"].shape != (B, width)
        if fresh:
            mk = lambda *s: torch.empty(*s, dtype=torch.int32, device=logits.device)
            out = dict(best=mk(B), accept_len=mk(B), next_token=mk(B), tokens=mk(B, width), indices=mk(B, width))
        if want_argmax and "node_argmax" not in out:
            out["node_argmax"] = torch.empty(B, T, dtype=torch.int32, device=logits.device)
        a.out_best_dev, a.out_accept_len_dev, a.out_next_token_dev = \
            out["best"].data_ptr(), out["accept_len"].data_ptr(), out["next_token"].data_ptr()
        a.out_tokens_dev, a.out_indices_dev = out["tokens"].data_ptr(), out["indices"].data_ptr()
        a.out_node_argmax_dev = out["node_argmax"].data_ptr() if want_argmax else None
        if want_topk and ("topk" not in out or out["topk"].shape[:2] != (B, T)):
            out["topk"] = torch.empty(B, T, 8, dtype=torch.int32, device=logits.device)
        a.out_topk_dev = out["topk"].data_ptr() if want_topk else None
        if recycle is not None:
            a.recycle_table_dev, a.recycle_owner_dev = recycle.table.data_ptr(), recycle.owner.data_ptr()
        else:
            a.recycle_table_dev, a.recycle_owner_dev = None, None
        with torch.cuda.device(self.device):
            K.check(K.lib().samd_verify_compact(self._h, C.byref(a), K.stream_ptr()), "samd_verify_compact")
        # remember the argument block for the fast path (keyed on the caller-provided `out`, if any)
        self._last_key = key[:10] + (out["tokens"].data_ptr(),) + key[11:]
        self._last_out = out
        return out

    def verify_sample(self, logits: torch.Tensor, tree_tokens: torch.Tensor, retrieve: Optional[torch.Tensor],
                      temperature: float, top_p: float, top_k: int, seeds: torch.Tensor, offsets: torch.Tensor,
                      n_paths: Optional[torch.Tensor] = None, want_sample_p: bool = False) -> dict:
        """Typical-acceptance verification + the draw of the next token (samd/utils.py:142-184, :85-88) for a batch:
        one launch, one CTA per request.  `seeds` / `offsets`: int64 CUDA tensors [B] - the Philox stream of every request
        (include/samd_b200.h states the contract); `offsets` is advanced in place by the draws used."""
        assert logits.is_cuda and logits.dim() == 3 and logits.stride(2) == 1
        B, T, V = logits.shape
        dt = {torch.bfloat16: K.DTYPE_BF16, torch.float16: K.DTYPE_FP16, torch.float32: K.DTYPE_FP32}.get(logits.dtype)
        if dt is None:
            raise K.SamdError(f"unsupported logits dtype {logits.dtype} (bf16 / fp16 / fp32)")
        _i32(tree_tokens)
        assert tree_tokens.shape == (B, T) and seeds.dtype == torch.int64 and offsets.dtype == torch.int64
        assert seeds.is_cuda and offsets.is_cuda and seeds.numel() == B and offsets.numel() == B
        a = K.SampleArgs()
        a.logits_dev, a.dtype, a.batch, a.n_nodes, a.vocab = logits.data_ptr(), dt, B, T, V
        a.batch_stride, a.row_stride = logits.stride(0), logits.stride(1)
        a.tree_tokens_dev = tree_tokens.data_ptr()
        if retrieve is not None:
            _i32(retrieve)
            if retrieve.dim() == 2:
                a.n_paths, a.depth, a.retrieve_batch_stride = retrieve.shape[0], retrieve.shape[1], 0
            else:
                a.n_paths, a.depth, a.retrieve_batch_stride = retrieve.shape[1], retrieve.shape[2], retrieve.stride(0)
            a.retrieve_dev, width = retrieve.data_ptr(), a.depth
        else:
            a.retrieve_dev, a.n_paths, a.depth, a.retrieve_batch_stride, width = None, 1, T, 0, T
        a.n_paths_dev = K.ptr(_i32(n_paths)) if n_paths is not None else None
        a.temperature, a.top_p, a.top_k = float(temperature), float(top_p), int(top_k)
        a.seeds_dev, a.offsets_dev = seeds.data_ptr(), offsets.data_ptr()
        mk = lambda *s: torch.empty(*s, dtype=torch.int32, device=logits.device)
        out = dict(best=mk(B), accept_len=mk(B), next_token=mk(B), tokens=mk(B, width), indices=mk(B, width))
        a.out_best_dev, a.out_accept_len_dev, a.out_next_token_dev = out["best"].data_ptr(), out["accept_len"].data_ptr(), out["next_token"].data_ptr()
        a.out_tokens_dev, a.out_indices_dev = out["tokens"].data_ptr(), out["indices"].data_ptr()
        if want_sample_p:
            out["sample_p"] = torch.empty(B, V, dtype=torch.float32, device=logits.device)
            a.out_sample_p_dev = out["sample_p"].data_ptr()
        else:
            a.out_sample_p_dev = None
        with torch.cuda.device(self.device):
            K.check(K.lib().samd_verify_sample(C.byref(a), K.stream_ptr()), "samd_verify_sample")
        return out

    def close(self):
        if self._h:
            K.lib().samd_verify_destroy(self._h)
            self._h = K.vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class RecycleTable:
    """Token-Recycle successor table on the device (samd/tree_model/token_recycle/token_recycle.py:18-63):
    table[token] = the 8 most likely next tokens the LM last predicted after `token` (-1 row = no entry), plus the
    static draft tree it fills.  Updated inside the verify launch (Verifier.verify(recycle=...)) or from any
    [N, V] logits block (update()); gen_tree() is TokenRecycle.gen_draft for a batch."""

    def __init__(self, tree: List[List[int]], vocab: Optional[int] = None, device: Optional[torch.device] = None):
        n = len(tree)
        parent, rank = [0] * n, [0] * n
        for node, childs in enumerate(tree):
            for j, c in enumerate(childs):
                if not node < c < n:
                    raise K.SamdError("RecycleTable: children must be numbered after their parent")
                parent[c], rank[c] = node, j
        self.tree, self.n_nodes = tree, n
        self._parent_host, self._rank_host = parent, rank
        self.table = self.owner = None
        self.vocab = 0
        self._ver = None
        if vocab is not None:
            self.ensure(vocab, device)

    def ensure(self, vocab: int, device=None):
        if self.table is not None:
            if vocab != self.vocab:
                raise K.SamdError(f"RecycleTable: vocabulary changed from {self.vocab} to {vocab}")
            return
        K.require_device()
        self.device = torch.device(device if device is not None else "cuda")
        self.vocab = int(vocab)
        self.table = torch.full((self.vocab, 8), -1, dtype=torch.int32, device=self.device)
        self.owner = torch.full((self.vocab,), -1, dtype=torch.int32, device=self.device)
        self.parent = torch.tensor(self._parent_host, dtype=torch.int32, device=self.device)
        self.rank = torch.tensor(self._rank_host, dtype=torch.int32, device=self.device)

    def update(self, tokens: torch.Tensor, logits: torch.Tensor) -> torch.Tensor:
        """table[tokens[i]] = top-8 of logits[i] for i in order (last occurrence of a token wins); [N] and [N, V].
        One launch: every row is a one-node request of the verify kernel.  Returns the [N, 8] top-8 indices."""
        assert logits.dim() == 2 and tokens.numel() == logits.shape[0]
        N, V = logits.shape
        self.ensure(V, logits.device)
        if self._ver is None or self._ver_cap < N:
            self._ver_cap = max(N, 256)
            self._ver = Verifier(self._ver_cap, 1, self.device)
        out = self._ver.verify(logits.view(N, 1, V), _i32(tokens.to(torch.int32).contiguous().view(N, 1)), None, recycle=self)
        return out["topk"].view(N, 8)

    def gen_tree(self, start_tok: torch.Tensor, types: Optional[torch.Tensor] = None, only_type: int = 0,
                 out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """[B, n_nodes] tree tokens: node 0 = start_tok[b], node c = table[token(parent(c))][rank(c)] or 0."""
        if self.table is None:
            raise K.SamdError("RecycleTable.gen_tree before the vocabulary is known (ensure(vocab) or an update first)")
        B = start_tok.numel()
        if out is None:
            out = torch.zeros(B, self.n_nodes, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            K.check(K.lib().samd_recycle_gen_tree(self.table.data_ptr(), self.vocab, self.parent.data_ptr(), self.rank.data_ptr(),
                                                  self.n_nodes, _i32(start_tok).data_ptr(), K.ptr(types), int(only_type), B,
                                                  out.data_ptr(), K.stream_ptr()), "samd_recycle_gen_tree")
        return out

    def as_dict(self) -> dict:
        """The reference's `cache` view: {token: [8 successors]} for every token with an entry."""
        if self.table is None:
            return {}
        t = self.table.cpu()
        have = (t[:, 0] >= 0).nonzero().flatten().tolist()
        return {k: t[k].tolist() for k in have}


def launch_count() -> int:
    return int(K.lib().samd_launch_count())
