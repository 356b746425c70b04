"""Batched (B > 1) speculative decode loop on top of the C ABI - SURVEY.md section 8f row 3.

The reference hard-wires batch size 1 (samd/samd_model.py:240).  Its per-request logic is applied here to B
requests in lockstep, with everything that the reference does on the host kept on the device:

    prefill (ragged prompts, right padded)                      -> DraftModel.update for every request
    loop:  samd_step            accepted tokens in, drafts out   (one launch for the whole batch)
           LM forward           [B, n_predicts] draft tokens, per-request positions, per-request KV offsets
           samd_verify_compact  accept lengths, accepted tokens, next tokens, cache_len += accept_len
           one tiny device->host read (all-finished flag) per step

Drafts are sequences of `n_predicts` tokens (the samd flavour's sequence type).  A request whose suffix match is
below `len_threshold` - where the reference falls back to its tree model - either simply verifies its start token
(draft = [start, pad...], the default) or, with `tree=<children lists>`, drafts the reference's Token-Recycle tree
(samd/tree_model/token_recycle/token_recycle.py) from a device-side successor table that the verify launch itself
keeps up to date.  In that mode every request carries T = max(n_predicts, len(tree)) nodes: a sequence request is
a chain (one path), a tree request uses the tree's ancestor mask and path table; node counts, path counts, masks,
positions and path tables are selected per request on the device, and samd_verify_compact moves the accepted
rows into place (cache.py:118-133).  Greedy verification makes any draft lossless, so the output stream equals
plain greedy decoding token for token.

BatchedSamOnlyDecoder runs the same loop with the samd_sam_only flavour's drafts: per-request variable-length
sequences and static-SAM trees, assembled into uniform batch buffers on the device by samd_draft_assemble.
"""
from __future__ import annotations

from typing import List, Optional, Sequence

import torch
from transformers.cache_utils import Cache, CacheLayerMixin

from . import _cabi as K
from . import engine as E

_cabi = K                       # (BatchedSamOnlyDecoder takes a parameter named K)


class _Layer(CacheLayerMixin):
    is_compileable = False
    is_sliding = False

    def __init__(self, parent, idx):
        super().__init__()
        self.parent, self.idx = parent, idx
        self.is_initialized = True

    def lazy_initialization(self, key_states, value_states):
        pass

    def update(self, key_states, value_states, *args, **kwargs):
        return self.parent.write(key_states, value_states, self.idx)

    def get_mask_sizes(self, query_length):
        return self.parent.kv_len, 0

    def get_seq_length(self):
        return 0

    def get_max_cache_shape(self):
        return self.parent.max_len

    def reset(self):
        pass


class RaggedKVCache(Cache):
    """[2L, B, H_kv, max_len, D_h] with a device-side length per request (SamdStaticCache generalised to B > 1):
    new rows are written at cache_len[b] + t."""

    def __init__(self, config, batch, max_len, dtype, device):
        L = config.num_hidden_layers
        super().__init__(layers=[_Layer(self, i) for i in range(L)])
        heads = getattr(config, "num_key_value_heads", None) or config.num_attention_heads
        dh = getattr(config, "head_dim", None) or config.hidden_size // config.num_attention_heads
        self.kv = torch.zeros(2 * L, batch, heads, max_len, dh, dtype=dtype, device=device)
        self.n_layers, self.batch, self.max_len = L, batch, max_len
        self.cache_len = torch.zeros(batch, dtype=torch.int32, device=device)
        self.kv_len = 0                 # key length the current forward attends over
        self.rows = None                # [B, T] absolute row of every new token in the current forward
        self._bidx = torch.arange(batch, device=device)[:, None]

    def begin(self, n_new: int, kv_len: int):
        # (clamped: a finished request still rides along in the batch; its rows may be written past its end, never past
        # the cache)
        self.rows = (self.cache_len.long()[:, None] + torch.arange(n_new, device=self.kv.device)[None, :]).clamp_(max=self.max_len - 1)
        self.kv_len = kv_len

    def write(self, k, v, layer):
        kc, vc = self.kv[layer], self.kv[self.n_layers + layer]
        kc[self._bidx, :, self.rows] = k.transpose(1, 2)
        vc[self._bidx, :, self.rows] = v.transpose(1, 2)
        return kc[:, :, :self.kv_len], vc[:, :, :self.kv_len]

    def get_seq_length(self, layer_idx=0):
        return 0


class BatchedSamdDecoder:
    def __init__(self, lm, batch: int, max_cache_len: int, n_predicts: int = 16, len_bias: int = 5, len_threshold: int = 5,
                 static: Optional[E.StaticSamDevice] = None, eos_token_id: Optional[int] = None, max_tokens: int = 16384,
                 dtype=torch.float16, device="cuda", tree: Optional[List[List[int]]] = None):
        self.lm, self.B, self.T = lm, batch, n_predicts
        self.n_seq = n_predicts
        self.device, self.dtype, self.eos = torch.device(device), dtype, eos_token_id
        self.cache = RaggedKVCache(lm.config, batch, max_cache_len, dtype, self.device)
        self.dyn = E.DynSamBatch(batch, max_tokens, self.device)
        self.eng = E.DraftEngine(self.dyn, static, K.FLAVOUR_SAMD, n_predicts=n_predicts, len_bias=len_bias,
                                 len_threshold=len_threshold)
        self.tree = tree
        if tree is not None:
            self._init_tree(tree)
        self.ver = E.Verifier(batch, self.T, self.device)
        self._ar = torch.arange(self.T, device=self.device)

    def _init_tree(self, tree):
        """Per-type tables, selected per request each step: ancestor masks, depths, path tables."""
        from . import synth
        dev, n_tree, n_seq = self.device, len(tree), self.n_seq
        T = self.T = max(n_seq, n_tree)
        self.table = E.RecycleTable(tree, self.lm.config.vocab_size, dev)
        parent = self.table._parent_host
        depth = [0] * n_tree
        for i in range(1, n_tree):
            depth[i] = depth[parent[i]] + 1
        anc = torch.eye(T, dtype=torch.bool)
        for i in range(n_tree):
            j = i
            while j != 0:
                j = parent[j]
                anc[i, j] = True
        chain = torch.eye(T, dtype=torch.bool)
        chain[:n_seq, :n_seq] = torch.tril(torch.ones(n_seq, n_seq, dtype=torch.bool))
        self._allow = torch.stack([chain, anc]).to(dev)                         # [2, T, T] (0 = sequence, 1 = tree)
        pos = torch.zeros(2, T, dtype=torch.long)
        pos[0, :n_seq] = torch.arange(n_seq)
        pos[1, :n_tree] = torch.tensor(depth)
        self._pos = pos.to(dev)
        ri = synth.tree_retrieve_indices(tree)                                   # [P, D_tree], -1 padded
        P, D = ri.shape[0], max(ri.shape[1], n_seq)
        ret = torch.full((2, P, D), -1, dtype=torch.int32)
        ret[0, 0, :n_seq] = torch.arange(n_seq, dtype=torch.int32)
        ret[1, :, :ri.shape[1]] = torch.as_tensor(ri, dtype=torch.int32)
        self._ret = ret.to(dev)
        self._n_nodes = torch.tensor([n_seq, n_tree], dtype=torch.int32, device=dev)
        self._n_paths = torch.tensor([1, P], dtype=torch.int32, device=dev)
        self._tree_tokens = torch.zeros(self.B, n_tree, dtype=torch.int32, device=dev)
        self.ver_bound = False

    def _mask(self, n_new: int, kv_len: int, base: torch.Tensor) -> torch.Tensor:
        """[B, 1, n_new, kv_len] additive mask: token t of request b sees keys j <= base[b] + t."""
        j = torch.arange(kv_len, device=self.device)[None, None, :]
        lim = (base.long()[:, None] + torch.arange(n_new, device=self.device)[None, :])[:, :, None]
        m = torch.zeros(self.B, n_new, kv_len, dtype=self.dtype, device=self.device)
        m.masked_fill_(j > lim, torch.finfo(self.dtype).min)
        return m[:, None]

    def _tree_step(self, start, kv_len, res):
        """One decode step with per-request draft shapes: sequence (chain) or Token-Recycle tree."""
        B, T, dev = self.B, self.T, self.device
        is_tree = (self.eng.out_type == K.DRAFT_TREE_MODEL)
        kind = is_tree.long()                                                      # 0 = sequence, 1 = tree
        self.table.gen_tree(start, types=self.eng.out_type, only_type=K.DRAFT_TREE_MODEL, out=self._tree_tokens)
        draft = torch.zeros(B, T, dtype=torch.int32, device=dev)
        draft[:, :self.n_seq] = self.eng.draft
        draft[:, 0] = start
        nt = self._tree_tokens.shape[1]
        draft[:, :nt] = torch.where(is_tree[:, None], self._tree_tokens, draft[:, :nt])
        if nt < T:
            draft[:, nt:] = torch.where(is_tree[:, None], torch.zeros_like(draft[:, nt:]), draft[:, nt:])
        base = self.cache.cache_len
        pos = base.long()[:, None] + self._pos[kind]
        # [B, 1, T, kv_len]: the past up to base[b], then the node's ancestors (chain or tree) at base[b] + j
        j = torch.arange(kv_len, device=dev)[None, None, :]
        rel = j - base.long()[:, None, None]                                       # [B, 1, kv_len] -> column's node id
        allow = self._allow[kind]                                                  # [B, T, T]
        in_new = (rel >= 0) & (rel < T)
        node_ok = torch.gather(allow, 2, rel.clamp(0, T - 1).expand(B, T, kv_len))
        ok = (rel < 0) | (in_new & node_ok)
        mask = torch.zeros(B, T, kv_len, dtype=self.dtype, device=dev)
        mask.masked_fill_(~ok, torch.finfo(self.dtype).min)
        logits = self.lm(input_ids=draft.long(), position_ids=pos, past_key_values=self.cache,
                         attention_mask=mask[:, None]).logits
        if not self.ver_bound:
            self.ver.bind_kv([self.cache.kv[i] for i in range(self.cache.kv.shape[0])])
            self.ver_bound = True
        return self.ver.verify(logits.contiguous(), draft, self._ret[kind].contiguous(), cache_len=self.cache.cache_len,
                               move_kv=True, n_nodes=self._n_nodes[kind].contiguous(), n_paths=self._n_paths[kind].contiguous(),
                               out=res, recycle=self.table)

    def _draft_forward_verify(self, kv_len: int) -> dict:
        """Drafts in, LM forward, fused verify: the part of a step that depends on the draft flavour."""
        st, T, cache = self._st, self.T, self.cache
        self.eng.step(st["acc_tokens"], st["acc_count"], st["start"])              # update(accepted) + lookup(start): one launch
        cache.begin(T, kv_len)
        if self.tree is not None:
            return self._tree_step(st["start"], kv_len, st["res"])
        draft = self.eng.draft
        draft[:, 0] = st["start"]                                                  # short matches verify the start token only
        pos = cache.cache_len.long()[:, None] + self._ar[None, :]
        logits = self.lm(input_ids=draft.long(), position_ids=pos, past_key_values=cache,
                         attention_mask=self._mask(T, kv_len, cache.cache_len)).logits
        return self.ver.verify(logits.contiguous(), draft, None, cache_len=cache.cache_len, out=st["res"])

    # ---- one decode step, entirely on the device (no host read anywhere: it is what gets captured in a CUDA graph) ----
    def _step_body(self, kv_len: int, max_new_tokens: int):
        st, T = self._st, self.T
        cache = self.cache
        # a request whose step could run past the cache is finished (samd_model.py:251-254)
        st["done"].logical_or_(cache.cache_len + T > cache.max_len)
        saved_len = cache.cache_len.clone()
        res = st["res"] = self._draft_forward_verify(kv_len)
        self._commit(res, saved_len, max_new_tokens)

    def _commit(self, res: dict, saved_len: torch.Tensor, max_new_tokens: int):
        """EOS truncation, emission, cache lengths, the next step's inputs, history and the host flag."""
        st, cache = self._st, self.cache
        done = st["done"]
        n_acc = torch.where(done, torch.zeros_like(res["accept_len"]), res["accept_len"])
        ar = self._ar[:res["tokens"].shape[1]]
        if self.eos is not None:                                                   # truncate at the first EOS (samd_model.py:257-263)
            is_eos = (res["tokens"] == self.eos) & (ar[None, :] < n_acc[:, None])
            first = torch.where(is_eos.any(1), is_eos.int().argmax(1).int() + 1, n_acc)
            done.logical_or_(is_eos.any(1))
            n_acc = torch.minimum(n_acc, first)
        room = (max_new_tokens - st["out_len"]).clamp(min=0)
        n_emit = torch.minimum(n_acc, room)
        out = st["out"]
        cols = st["out_len"].long()[:, None] + ar[None, :]
        keep = ar[None, :] < n_emit[:, None]
        out.scatter_(1, torch.where(keep, cols, torch.full_like(cols, out.shape[1] - 1)),
                     torch.where(keep, res["tokens"], torch.zeros_like(res["tokens"])))
        st["out_len"].add_(n_emit)
        done.logical_or_(st["out_len"] >= max_new_tokens)
        cache.cache_len.copy_(saved_len + n_acc)                                   # finished requests stop advancing
        st["acc_tokens"].copy_(res["tokens"])
        st["acc_count"].copy_(n_acc)
        st["start"].copy_(res["next_token"])
        st["hist"].index_copy_(0, st["step"], n_acc[None, :])
        st["step"].add_(1)
        # what the host reads every `check_every` steps: [all finished?, longest cache]
        st["flag"][0] = done.all().to(torch.int32)
        st["flag"][1] = cache.cache_len.max()

    def _prefill_hook(self, ids: torch.Tensor, lens: torch.Tensor, logits: torch.Tensor):
        """After the prompt's forward and automaton update: TokenRecycle.update over the prompt rows (tree mode)."""
        if self.tree is not None:
            n_max = ids.shape[1]
            valid = torch.arange(n_max, device=ids.device)[None, :] < lens[:, None]
            self.table.update(ids[valid].to(torch.int32), logits[valid])
            if not self.ver_bound:
                self.ver.bind_kv([self.cache.kv[i] for i in range(self.cache.kv.shape[0])])
                self.ver_bound = True

    def _extra_state(self, mk) -> dict:
        """Step state of a subclass, kept with the rest (persistent, snapshotted around a capture, zeroed per call)."""
        return {}

    @torch.inference_mode()
    def generate(self, prompts: Sequence[Sequence[int]], max_new_tokens: int, graph: bool = True, check_every: int = 4):
        """Lossless batched speculative decoding.  The decode step has no host synchronisation in it: it is captured
        once per key-length bucket (64 positions) as a CUDA graph and replayed; the host reads a two-word flag (all
        finished / longest cache) once every `check_every` steps - 1 / check_every host syncs per step - and sizes
        the next steps' key length from that bound.  A finished batch may therefore run up to check_every - 1 idle
        steps (every request done: nothing is emitted).  graph=False runs the same body eagerly."""
        B, T, dev = self.B, self.T, self.device
        assert len(prompts) == B
        lens = torch.tensor([len(p) for p in prompts], dtype=torch.int32, device=dev)
        n_max = int(lens.max())
        # the reference stops a request before a step that could run past the cache (samd_model.py:251-254); here the
        # prompt itself must leave room for one step, and a request that gets within one step of the end is finished
        if n_max + T > self.cache.max_len:
            raise K.SamdError(f"prompt of {n_max} tokens + one decode step of {T} does not fit max_cache_len={self.cache.max_len}")
        if n_max + max_new_tokens + T > self.dyn.max_tokens:
            raise K.SamdError(f"prompt + max_new_tokens + one step = {n_max + max_new_tokens + T} exceeds the automaton "
                              f"capacity max_tokens={self.dyn.max_tokens}")
        ids = torch.zeros(B, n_max, dtype=torch.long, device=dev)
        for b, p in enumerate(prompts):
            ids[b, :len(p)] = torch.as_tensor(p, dtype=torch.long)
        # ---- prefill ------------------------------------------------------------------------
        self.eng.reset()
        self.cache.cache_len.zero_()
        self.cache.begin(n_max, n_max)
        pos = torch.arange(n_max, device=dev)[None, :].expand(B, -1)
        logits = self.lm(input_ids=ids, position_ids=pos, past_key_values=self.cache,
                         attention_mask=self._mask(n_max, n_max, torch.zeros(B, dtype=torch.int32, device=dev))).logits
        self.cache.cache_len.copy_(lens)
        self.eng.step(ids.to(torch.int32).contiguous(), lens, None)                # DraftModel.update(prompt), ragged counts
        self._prefill_hook(ids, lens, logits)
        max_steps = max_new_tokens + check_every + 1
        width = T if self.tree is None else self._ret.shape[2]
        first_tok = logits[torch.arange(B, device=dev), lens.long() - 1].argmax(-1).to(torch.int32)
        key = (max_new_tokens, max_steps, width)
        if getattr(self, "_st_key", None) != key:
            # the step's state lives in tensors that persist across generate() calls: the captured graphs refer to them
            mk = lambda *sh: torch.zeros(*sh, dtype=torch.int32, device=dev)
            self._st = dict(start=mk(B), acc_tokens=mk(B, width), acc_count=mk(B), out=mk(B, max_new_tokens + T), out_len=mk(B),
                            done=torch.zeros(B, dtype=torch.bool, device=dev), hist=mk(max_steps, B),
                            step=torch.zeros(1, dtype=torch.long, device=dev), flag=mk(2), res=None, **self._extra_state(mk))
            self._st_key, self._graphs = key, {}
        else:
            for k, v in self._st.items():
                if k not in ("start", "res"):
                    v.zero_()
        self._st["start"].copy_(first_tok)
        flag_host = torch.zeros(2, dtype=torch.int32).pin_memory()
        # ---- decode ---------------------------------------------------------------------------
        max_accept = width                     # the most one step can add to a request's cache
        kv_hi, since, steps, syncs = n_max, 0, 0, 0
        graphs = self._graphs
        self.last_graphed = False
        while steps < max_steps - 1:
            kv_len = min((kv_hi + since * max_accept + T + 63) // 64 * 64, self.cache.max_len)
            if graph:
                g = graphs.get(kv_len)
                if g is None:
                    # warm-up run on a side stream (allocations, lazy initialisation), state restored, then the capture
                    snap = {k: (v.clone() if torch.is_tensor(v) else v) for k, v in self._st.items() if k != "res"}
                    snap_len = self.cache.cache_len.clone()
                    snap_dyn = E.DynSamBatch(B, self.dyn.max_tokens, dev)
                    snap_dyn.copy_from(self.dyn)
                    snap_cur = self.eng.static_cursor.clone() if self.eng.static_cursor is not None else None
                    snap_tab = (self.table.table.clone(), self.table.owner.clone()) if self.tree is not None else None
                    side = torch.cuda.Stream(dev)
                    side.wait_stream(torch.cuda.current_stream(dev))
                    with torch.cuda.stream(side):
                        self._step_body(kv_len, max_new_tokens)
                    torch.cuda.current_stream(dev).wait_stream(side)

                    def restore():
                        for k, v in snap.items():
                            if torch.is_tensor(v):
                                self._st[k].copy_(v)
                        self.cache.cache_len.copy_(snap_len)
                        self.dyn.copy_from(snap_dyn)
                        if snap_cur is not None:
                            self.eng.static_cursor.copy_(snap_cur)
                        if snap_tab is not None:
                            self.table.table.copy_(snap_tab[0])
                            self.table.owner.copy_(snap_tab[1])

                    restore()
                    torch.cuda.synchronize(dev)
                    try:
                        g = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(g):
                            self._step_body(kv_len, max_new_tokens)
                        graphs[kv_len] = g
                        self.last_graphed = True
                    except Exception:                      # an LM whose forward cannot be captured: same body, eagerly
                        graph = False
                        torch.cuda.synchronize(dev)
                    restore()                              # (capture does not run the work; the warm-up did)
                    snap_dyn.close()
                if graph:
                    graphs[kv_len].replay()
                    self.last_graphed = True
            if not graph:
                self._step_body(kv_len, max_new_tokens)
            steps += 1
            since += 1
            if since == check_every:
                flag_host.copy_(self._st["flag"], non_blocking=True)
                torch.cuda.current_stream(dev).synchronize()                       # the host sync: once per check_every steps
                syncs += 1
                if int(flag_host[0]):
                    break
                kv_hi, since = int(flag_host[1]), 0
        st = self._st
        lens_out = st["out_len"].tolist()
        rows = st["out"].tolist()
        hist = st["hist"][:steps].t().tolist()
        n_live = max((max((i + 1 for i, a in enumerate(h) if a), default=0) for h in hist), default=0)
        return ([rows[b][:lens_out[b]] for b in range(B)],
                dict(steps=n_live, steps_run=steps, host_syncs=syncs, graphed=self.last_graphed, graphs=len(graphs),
                     accept_lengths=[h[:n_live] for h in hist]))


class BatchedSamOnlyDecoder(BatchedSamdDecoder):
    """Batched decoding with the `samd_sam_only` flavour (samd_sam_only/samd_model.py:117-157 for B requests in lockstep):
    every request drafts either a dynamic-automaton sequence of min(max_predicts, 1 + int(match * alpha)) tokens or, when
    a static automaton built with counts is bound and wins by more than `len_bias`, the static SAM's best-first tree of up
    to max_predicts nodes (K children per level).  One step, all on the device:

        samd_step              update(accepted) + lookup(start): per-request type, draft, draft_len
        samd_static_tree_draft the trees of the requests typed DRAFT_STATIC_TREE (static automaton only)
        samd_draft_assemble    uniform [B, T] tokens / position ids, [B, T, kv_len] additive mask, [B, P, D] path table,
                               node and path counts; finished requests get a one-node draft with no path
        LM forward             position_ids and attention_mask = mask[:, None]
        samd_verify_compact    accept lengths, accepted tokens, next tokens, the accepted KV rows moved into place

    T = P = D = max_predicts.  The rest of the loop (prefill, one CUDA graph per key-length bucket, the commit, one host
    read per `check_every` steps) is BatchedSamdDecoder's.  stats["tree_steps"] counts the request-steps of live requests
    that drafted a static tree.

    Known corner, inherited from the reference (SURVEY Appendix A9): a -1 pad column of a path selects token 0, so it is
    "accepted" when the compared row's argmax is token 0, and the KV move then copies row cache_len - 1.  The batched path
    table is D wide while a reference tree is only as wide as its own deepest path (and a reference sequence as long as
    its draft), so here pads beyond a request's own width can be compared too - only after every real node of the path
    was accepted, i.e. when the LM's greedy next token is 0."""

    def __init__(self, lm, batch: int, max_cache_len: int, max_predicts: int = 40, alpha: float = 4.0, K: int = 8,
                 len_bias: int = 5, static: Optional[E.StaticSamDevice] = None, eos_token_id: Optional[int] = None,
                 max_tokens: int = 16384, dtype=torch.float16, device="cuda"):
        if static is not None and not static.with_counts:
            raise _cabi.SamdError("BatchedSamOnlyDecoder: the static automaton must be built with_counts=True "
                                  "(the sam_only tree drafter reads its occurrence counts and top-8 successors)")
        if not 1 <= max_predicts <= 128:
            raise _cabi.SamdError(f"BatchedSamOnlyDecoder: max_predicts must be in [1, 128], got {max_predicts}")
        self.lm, self.B, self.T = lm, batch, max_predicts
        self.device, self.dtype, self.eos = torch.device(device), dtype, eos_token_id
        self.tree, self.K_top = None, int(K)
        self.cache = RaggedKVCache(lm.config, batch, max_cache_len, dtype, self.device)
        self.dyn = E.DynSamBatch(batch, max_tokens, self.device)
        self.eng = E.DraftEngine(self.dyn, static, _cabi.FLAVOUR_SAM_ONLY, n_predicts=max_predicts, len_bias=len_bias,
                                 alpha=alpha)
        self.ver = E.Verifier(batch, max_predicts, self.device)
        self.ver.bind_kv([self.cache.kv[i] for i in range(self.cache.kv.shape[0])])
        self._ar = torch.arange(max_predicts, device=self.device)
        # the assembled buffers persist: the captured graphs refer to them.  The mask of a kv_len bucket is the leading
        # [B, T, kv_len] block of one flat allocation sized for the whole cache.
        T, dev = max_predicts, self.device
        mk = lambda *s: torch.zeros(*s, dtype=torch.int32, device=dev)
        self.buf = dict(tokens=mk(batch, T), position_ids=torch.zeros(batch, T, dtype=torch.long, device=dev),
                        n_nodes=mk(batch), n_paths=mk(batch), retrieve=mk(batch, T, T),
                        mask=torch.zeros(batch * T * max_cache_len, dtype=dtype, device=dev))

    def _extra_state(self, mk) -> dict:
        return dict(tree_steps=torch.zeros(1, dtype=torch.long, device=self.device))

    def mask_view(self, kv_len: int) -> torch.Tensor:
        return self.buf["mask"][:self.B * self.T * kv_len].view(self.B, self.T, kv_len)

    def _draft_forward_verify(self, kv_len: int) -> dict:
        st, T, cache, eng, buf = self._st, self.T, self.cache, self.eng, self.buf
        eng.step(st["acc_tokens"], st["acc_count"], st["start"])
        if eng.static is not None:
            eng.tree_draft(st["start"], K_top=self.K_top)
        st["tree_steps"].add_(((eng.out_type == _cabi.DRAFT_STATIC_TREE) & ~st["done"]).sum())
        mask = self.mask_view(kv_len)
        eng.assemble(cache.cache_len, buf["tokens"], buf["position_ids"], buf["n_nodes"], buf["n_paths"], buf["retrieve"],
                     mask, done=st["done"])
        cache.begin(T, kv_len)
        logits = self.lm(input_ids=buf["tokens"].long(), position_ids=buf["position_ids"], past_key_values=cache,
                         attention_mask=mask[:, None]).logits
        return self.ver.verify(logits.contiguous(), buf["tokens"], buf["retrieve"], cache_len=cache.cache_len, move_kv=True,
                               n_nodes=buf["n_nodes"], n_paths=buf["n_paths"], out=st["res"])

    @torch.inference_mode()
    def generate(self, prompts: Sequence[Sequence[int]], max_new_tokens: int, graph: bool = True, check_every: int = 4):
        """BatchedSamdDecoder.generate; stats also carry "tree_steps"."""
        out, stats = super().generate(prompts, max_new_tokens, graph=graph, check_every=check_every)
        stats["tree_steps"] = int(self._st["tree_steps"].item())
        return out, stats
