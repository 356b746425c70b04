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

generate() decodes exactly B prompts in lockstep.  serve() is continuous batching over the same loop: any number of
requests, each admitted into a slot as soon as the host sees that slot's request finished (prefill of the admitted
prompts alone, masked drafter reset, prompt ingestion with count 0 for every other request, the slot's state written in
place), so the graphs captured per key-length bucket stay valid and nothing waits for the longest request of a batch.
"""
from __future__ import annotations

from typing import Iterable, Iterator, List, Optional, Sequence, Union

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
        self._slots = None              # [n, 1] requests of a sub-batch forward (begin(slots=...)), None = the whole batch

    def begin(self, n_new: int, kv_len: int, slots: Optional[torch.Tensor] = None):
        """Set up the next forward.  By default it carries every request and writes its new rows at cache_len[b] + t.
        With `slots` (int64 [n]) it carries only those requests, in that order - a prefill of newly admitted requests:
        rows 0 .. n_new - 1 of those slots are written and attention reads those slots alone."""
        ar = torch.arange(n_new, device=self.kv.device)[None, :]
        if slots is None:
            # (clamped: a finished request still rides along in the batch; its rows may be written past its end, never
            # past the cache)
            self._slots = None
            self.rows = (self.cache_len.long()[:, None] + ar).clamp_(max=self.max_len - 1)
        else:
            self._slots = slots[:, None]
            self.rows = ar.expand(slots.numel(), -1)
        self.kv_len = kv_len

    def write(self, k, v, layer):
        kc, vc = self.kv[layer], self.kv[self.n_layers + layer]
        b = self._bidx if self._slots is None else self._slots
        kc[b, :, self.rows] = k.transpose(1, 2)
        vc[b, :, self.rows] = v.transpose(1, 2)
        if self._slots is None:
            return kc[:, :, :self.kv_len], vc[:, :, :self.kv_len]
        return kc[b[:, 0], :, :self.kv_len], vc[b[:, 0], :, :self.kv_len]

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
        """[n, 1, n_new, kv_len] additive mask (n = base.numel(), the batch or a sub-batch): token t of request b sees keys
        j <= base[b] + t."""
        j = torch.arange(kv_len, device=self.device)[None, None, :]
        lim = (base.long()[:, None] + torch.arange(n_new, device=self.device)[None, :])[:, :, None]
        m = torch.zeros(base.numel(), n_new, kv_len, dtype=self.dtype, device=self.device)
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
    def _step_body(self, kv_len: int):
        st, T = self._st, self.T
        cache = self.cache
        # a request whose step could run past the cache is finished (samd_model.py:251-254)
        st["done"].logical_or_(cache.cache_len + T > cache.max_len)
        saved_len = cache.cache_len.clone()
        res = st["res"] = self._draft_forward_verify(kv_len)
        self._commit(res, saved_len)

    def _commit(self, res: dict, saved_len: torch.Tensor):
        """EOS truncation, emission up to each slot's own limit, cache lengths, the next step's inputs, history and the
        host flag."""
        st, cache = self._st, self.cache
        done = st["done"]
        n_acc = torch.where(done, torch.zeros_like(res["accept_len"]), res["accept_len"])
        ar = self._ar[:res["tokens"].shape[1]]
        if self.eos is not None:                                                   # truncate at the first EOS (samd_model.py:257-263)
            is_eos = (res["tokens"] == self.eos) & (ar[None, :] < n_acc[:, None])
            first = torch.where(is_eos.any(1), is_eos.int().argmax(1).int() + 1, n_acc)
            done.logical_or_(is_eos.any(1))
            n_acc = torch.minimum(n_acc, first)
        room = (st["limit"] - st["out_len"]).clamp(min=0)
        n_emit = torch.minimum(n_acc, room)
        out = st["out"]
        cols = st["out_len"].long()[:, None] + ar[None, :]
        keep = ar[None, :] < n_emit[:, None]
        out.scatter_(1, torch.where(keep, cols, torch.full_like(cols, out.shape[1] - 1)),
                     torch.where(keep, res["tokens"], torch.zeros_like(res["tokens"])))
        st["out_len"].add_(n_emit)
        done.logical_or_(st["out_len"] >= st["limit"])
        cache.cache_len.copy_(saved_len + n_acc)                                   # finished requests stop advancing
        st["acc_tokens"].copy_(res["tokens"])
        st["acc_count"].copy_(n_acc)
        st["start"].copy_(res["next_token"])
        # per-slot history of live steps (a live step accepts >= 1 token): hist[b, hlen[b]] = n_acc[b]; a finished
        # request writes the spare last column
        hist, live = st["hist"], n_acc > 0
        col = torch.where(live, st["hlen"], hist.shape[1] - 1)
        hist.scatter_(1, col.long()[:, None], n_acc[:, None])
        st["hlen"].add_(live.to(torch.int32))
        # what the host reads every `check_every` steps: [done (B) | out_len (B) | longest cache]
        torch.cat((done.to(torch.int32), st["out_len"], cache.cache_len.max()[None]), out=st["flag"])

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

    def _extra_stats(self) -> dict:
        """Statistics of a subclass, read at the end of a call."""
        return {}

    # ---- the step state, and the CUDA graphs that refer to it -------------------------------------------------------
    def _init_state(self, max_limit: int):
        """Zeroed step state for requests of at most `max_limit` new tokens.  The tensors persist across calls (the
        captured graphs refer to them, and limits are per slot); they are reallocated, and the graphs dropped, only when
        a call needs longer outputs than any before."""
        B, T, dev = self.B, self.T, self.device
        width = T if self.tree is None else self._ret.shape[2]
        cap = getattr(self, "_st_cap", None)
        if cap is None or cap < max_limit:
            mk = lambda *sh: torch.zeros(*sh, dtype=torch.int32, device=dev)
            # out: a slot's tokens plus spare columns; hist: its live steps (each emits >= 1 token, so at most max_limit)
            # plus a spare column; hlen: its live-step count; limit: its max_new_tokens
            self._st = dict(start=mk(B), acc_tokens=mk(B, width), acc_count=mk(B), out=mk(B, max_limit + T), out_len=mk(B),
                            limit=mk(B), done=torch.zeros(B, dtype=torch.bool, device=dev), hist=mk(B, max_limit + 1),
                            hlen=mk(B), flag=mk(2 * B + 1), res=None, **self._extra_state(mk))
            self._st_cap, self._graphs = max_limit, {}
        else:
            for k, v in self._st.items():
                if k != "res":
                    v.zero_()

    def _advance(self, kv_len: int, graph: bool) -> bool:
        """One decode step at key length `kv_len`: the bucket's CUDA graph, captured first if it is new, or the same body
        eagerly.  Returns `graph`, False from then on when the LM's forward cannot be captured."""
        if graph:
            B, dev, graphs = self.B, self.device, self._graphs
            if kv_len not in graphs:
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
                    self._step_body(kv_len)
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
                        self._step_body(kv_len)
                    graphs[kv_len] = g
                    self.last_graphed = True
                except Exception:                          # an LM whose forward cannot be captured: same body, eagerly
                    graph = False
                    torch.cuda.synchronize(dev)
                restore()                                  # (capture does not run the work; the warm-up did)
                snap_dyn.close()
            if graph:
                graphs[kv_len].replay()
                self.last_graphed = True
                return True
        self._step_body(kv_len)
        return False

    # ---- admission: new requests into free slots, between two steps ---------------------------------------------------
    def _admit(self, reqs: List[tuple]) -> int:
        """Start the requests `reqs` = [(slot, prompt, limit)] in their (free) slots; returns the longest prompt.  Only
        the persistent state is written, in place, so the captured graphs stay valid."""
        dev = self.device
        n_max = max(len(p) for _, p, _ in reqs)
        ids = torch.zeros(len(reqs), n_max, dtype=torch.long)
        for i, (_, p, _) in enumerate(reqs):
            ids[i, :len(p)] = torch.as_tensor(p, dtype=torch.long)
        meta = torch.tensor([[r[0] for r in reqs], [len(r[1]) for r in reqs], [r[2] for r in reqs]], dtype=torch.long)
        ids, meta = ids.to(dev), meta.to(dev)
        slots, lens, limits = meta[0], meta[1].to(torch.int32), meta[2].to(torch.int32)
        logits = self._prefill_slots(ids, slots)
        self._ingest(ids, slots, lens, logits)
        self._set_slots(slots, lens, limits, logits)
        return n_max

    def _prefill_slots(self, ids: torch.Tensor, slots: torch.Tensor) -> torch.Tensor:
        """LM prefill of the admitted prompts alone ([n, n_max], right padded) into KV rows 0 .. n_max - 1 of their
        slots: the cost follows the admitted prompts, not the batch."""
        n, n_max = ids.shape
        self.cache.begin(n_max, n_max, slots=slots)
        pos = torch.arange(n_max, device=self.device)[None, :].expand(n, -1)
        return self.lm(input_ids=ids, position_ids=pos, past_key_values=self.cache,
                       attention_mask=self._mask(n_max, n_max, torch.zeros(n, dtype=torch.int32, device=self.device))).logits

    def _ingest(self, ids: torch.Tensor, slots: torch.Tensor, lens: torch.Tensor, logits: torch.Tensor):
        """The admitted requests' drafters: masked DraftModel.reset (automaton and static cursor), then
        DraftModel.update(prompt) in one launch with count 0 for every other request, then the prefill hook."""
        B, dev = self.B, self.device
        self.eng.reset(torch.zeros(B, dtype=torch.uint8, device=dev).index_fill_(0, slots, 1))
        tokens = torch.zeros(B, ids.shape[1], dtype=torch.int32, device=dev).index_copy_(0, slots, ids.to(torch.int32))
        counts = torch.zeros(B, dtype=torch.int32, device=dev).index_copy_(0, slots, lens)
        self.eng.step(tokens, counts, None)
        self._prefill_hook(ids, lens, logits)

    def _set_slots(self, slots: torch.Tensor, lens: torch.Tensor, limits: torch.Tensor, logits: torch.Tensor):
        """The admitted slots' step state: cache length, first start token (the prompt's greedy next token), limit, and
        zero emitted tokens / history."""
        st = self._st
        first = logits[torch.arange(slots.numel(), device=self.device), lens.long() - 1].argmax(-1).to(torch.int32)
        self.cache.cache_len.index_copy_(0, slots, lens)
        st["start"].index_copy_(0, slots, first)
        st["limit"].index_copy_(0, slots, limits)
        for k in ("acc_count", "out_len", "hlen"):
            st[k].index_fill_(0, slots, 0)
        st["done"].index_fill_(0, slots, False)

    # ---- the decode loop of generate() and serve() --------------------------------------------------------------------
    def _run(self, requests: Iterator[tuple], max_limit: int, graph: bool, check_every: int):
        """Decode the validated requests (index, prompt, limit) of `requests`, at most B at a time.  The decode step has
        no host synchronisation in it: it is captured once per key-length bucket (64 positions) as a CUDA graph and
        replayed.  Once every `check_every` steps the host reads [done | out_len | longest cache] in one copy; it then
        yields (index, tokens, accept_lengths, slot) for every request found finished (their rows in one more copy),
        admits queued requests into the free slots, and sizes the next steps' key length from the longest cache.  A
        finished request keeps its slot - riding along, emitting nothing - until that check.  Statistics go to
        self._run_stats."""
        B, T, dev = self.B, self.T, self.device
        self._init_state(max_limit)
        st = self._st
        run = self._run_id = getattr(self, "_run_id", 0) + 1
        self.eng.reset()
        self.cache.cache_len.zero_()
        st["done"].fill_(True)                                                     # an empty slot rides along finished
        owner = [None] * B                                                         # request index in each slot
        W, max_accept = st["out"].shape[1], st["acc_tokens"].shape[1]              # (the most one step adds to a cache)
        flag_host = torch.zeros(2 * B + 1, dtype=torch.int32).pin_memory()
        steps = syncs = since = admissions = live_steps = 0
        self.last_graphed = False

        def admit() -> int:
            nonlocal admissions
            reqs = []
            for b in range(B):
                if owner[b] is None:
                    r = next(requests, None)
                    if r is None:
                        break
                    owner[b] = r[0]
                    reqs.append((b, r[1], r[2]))
            admissions += len(reqs)
            return self._admit(reqs) if reqs else 0

        kv_hi = admit()
        while any(o is not None for o in owner):
            kv_len = min((kv_hi + since * max_accept + T + 63) // 64 * 64, self.cache.max_len)
            graph = self._advance(kv_len, graph)
            steps += 1
            since += 1
            if since < check_every:
                continue
            flag_host.copy_(st["flag"], non_blocking=True)
            torch.cuda.current_stream(dev).synchronize()                           # the host sync: once per check_every steps
            syncs += 1
            since = 0
            flag = flag_host.tolist()
            kv_hi = flag[2 * B]
            fin = [b for b in range(B) if owner[b] is not None and flag[b]]
            if fin:
                idx = torch.tensor(fin, device=dev)
                rows = torch.cat((st["out"][idx], st["hist"][idx], st["hlen"][idx, None]), 1).tolist()
                for b, r in zip(fin, rows):
                    i, owner[b] = owner[b], None
                    hist = r[W:W + r[-1]]
                    live_steps += len(hist)
                    yield i, r[:flag[B + b]], hist, b
                    if self._run_id != run:
                        raise K.SamdError("the decoder ran another generate() / serve() while this serve() was suspended")
            kv_hi = max(kv_hi, admit())
        self._run_stats = dict(steps_run=steps, host_syncs=syncs, graphed=self.last_graphed, graphs=len(self._graphs),
                               admissions=admissions, live_slot_steps=live_steps, **self._extra_stats())

    @torch.inference_mode()
    def generate(self, prompts: Sequence[Sequence[int]], max_new_tokens: int, graph: bool = True, check_every: int = 4):
        """Lossless batched speculative decoding of exactly B prompts in lockstep (request b in slot b), up to
        max_new_tokens each.  The host reads the finished flags once every `check_every` steps - 1 / check_every host
        syncs per step - so a finished batch may run up to check_every - 1 idle steps (every request done: nothing is
        emitted).  graph=False runs the same body eagerly.  Returns (tokens per request, stats); stats["accept_lengths"]
        holds every request's accepted tokens per step, padded with 0 to the longest request's `steps`."""
        B, T = self.B, self.T
        assert len(prompts) == B
        n_max = max(len(p) for p in prompts)
        # the reference stops a request before a step that could run past the cache (samd_model.py:251-254); here the
        # prompt itself must leave room for one step, and a request that gets within one step of the end is finished
        if n_max + T > self.cache.max_len:
            raise K.SamdError(f"prompt of {n_max} tokens + one decode step of {T} does not fit max_cache_len={self.cache.max_len}")
        if n_max + max_new_tokens + T > self.dyn.max_tokens:
            raise K.SamdError(f"prompt + max_new_tokens + one step = {n_max + max_new_tokens + T} exceeds the automaton "
                              f"capacity max_tokens={self.dyn.max_tokens}")
        out, acc = [None] * B, [None] * B
        for i, tokens, hist, _ in self._run(((i, p, max_new_tokens) for i, p in enumerate(prompts)), max_new_tokens,
                                            graph, check_every):
            out[i], acc[i] = tokens, hist
        n_live = max(len(a) for a in acc)
        s = self._run_stats
        return out, dict(steps=n_live, steps_run=s["steps_run"], host_syncs=s["host_syncs"], graphed=s["graphed"],
                         graphs=s["graphs"], accept_lengths=[a + [0] * (n_live - len(a)) for a in acc], **self._extra_stats())

    @torch.inference_mode()
    def serve(self, prompts: Iterable[Sequence[int]], max_new_tokens: Union[int, Sequence[int]], graph: bool = True,
              check_every: int = 4):
        """Continuous batching: decode any number of requests through the B slots, refilling a slot with the next queued
        request as soon as the host sees its request finished (once every `check_every` steps).  `prompts` is consumed
        lazily and in order; `max_new_tokens` is one limit for all or a sequence with one per request.  Yields
        (index, tokens, {"slot", "accept_lengths"}) per request in completion order; `tokens` are what generate() emits
        for that prompt, `accept_lengths` has one entry per live decode step.  A request is validated when it is pulled
        (SamdError naming its index).  self.serve_stats is set once the generator is exhausted: steps_run, host_syncs
        (flag reads), graphed, graphs, admissions, live_slot_steps (slot-steps of unfinished requests) and, for
        BatchedSamOnlyDecoder, tree_steps.  One call at a time: a generate() or serve() call while this generator is
        suspended ends it (it raises when resumed); an abandoned generator leaves the decoder usable."""
        self.serve_stats = None
        if hasattr(max_new_tokens, "__len__"):
            limits = [int(x) for x in max_new_tokens]
            max_limit = max(limits, default=1)
        else:
            limits, max_limit = None, int(max_new_tokens)
        for i, tokens, hist, slot in self._run(self._requests(prompts, max_new_tokens if limits is None else limits),
                                               max(max_limit, 1), graph, check_every):
            yield i, tokens, {"slot": slot, "accept_lengths": hist}
        self.serve_stats = dict(self._run_stats)

    def _requests(self, prompts: Iterable[Sequence[int]], limits: Union[int, List[int]]) -> Iterator[tuple]:
        """(index, prompt, limit) of every request, checked as it is pulled."""
        T, max_len, cap = self.T, self.cache.max_len, self.dyn.max_tokens
        for i, p in enumerate(prompts):
            if isinstance(limits, list):
                if i >= len(limits):
                    raise K.SamdError(f"request {i}: max_new_tokens has {len(limits)} values, fewer than the prompts")
                limit = limits[i]
            else:
                limit = limits
            n = len(p)
            if n == 0:
                raise K.SamdError(f"request {i}: empty prompt")
            if limit < 1:
                raise K.SamdError(f"request {i}: max_new_tokens must be >= 1, got {limit}")
            if n + T > max_len:
                raise K.SamdError(f"request {i}: prompt of {n} tokens + one decode step of {T} does not fit "
                                  f"max_cache_len={max_len}")
            if n + limit + T > cap:
                raise K.SamdError(f"request {i}: prompt + max_new_tokens + one step = {n + limit + T} exceeds the "
                                  f"automaton capacity max_tokens={cap}")
            yield i, p, limit


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
    read per `check_every` steps, generate() and serve()) is BatchedSamdDecoder's.  stats["tree_steps"] (and
    serve_stats["tree_steps"]) counts the request-steps of live requests that drafted a static tree.

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

    def _extra_stats(self) -> dict:
        return dict(tree_steps=int(self._st["tree_steps"].item()))

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
