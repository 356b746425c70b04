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
With a prefix pool (max_prefixes > 0, add_prefix) an admitted request whose prompt starts with a registered prefix copies
that prefix's KV rows, automaton and static cursor and prefills / ingests only the rest of its prompt.

generate(..., sampling=...) and serve(..., sampling=...) decode with sampling instead (SamplingParams: temperature, top-p,
top-k and a seed per request, as the reference's SamdGenerationConfig(greedy=False)): the verify step is
samd_verify_sample_requests with every slot's own processor and Philox stream, and the first token of a request is drawn
from the plain softmax of its prompt's last row.  A request's tokens depend only on its prompt, its parameters and its
seed - not on its slot, its neighbours, the batch size, graph or eager execution, check_every, or a prefix pool.

generate(..., logprobs=n) and serve(..., logprobs=n) also return every emitted token's log-probability (raw, or of the
penalized row with penalties=) and its n best alternatives (n in [0, 8]).  After the verify launch, one
samd_token_logprobs launch scores the accepted rows of the step's logits; each slot carries the log-probability of its start token (predicted by the previous step's last accepted row,
or at admission by the prompt's last row), and the commit writes them beside the tokens with the same truncation.

generate(..., penalties=...) and serve(..., penalties=...) apply repetition, presence and frequency penalties (Penalties,
one per request) before verification or sampling.  Each draft row is penalized from its own context - prompt, emitted
tokens and the draft tokens on its path - by one samd_apply_penalties launch between the LM forward and the verify
launch, so greedy verification stays lossless against plain penalized greedy decoding.  Every slot keeps a device count
table row (output counts, a bit for the prompt's tokens), filled at admission and by the commit.

generate(..., stop=...) and serve(..., stop=...) end a request at the earliest of its stop sequences (StopSequences: up
to 16 sequences of up to 16 token ids, matched against the output only).  One step accepts up to T tokens, so a sequence
may end inside a step or straddle two: after the EOS cut, one samd_stop_match launch in the commit finds each request's
earliest match among the tokens the step would emit (and the last 15 it emitted before), and the commit emits up to it.
Every request also gets a finish reason: "stop" (EOS or a stop sequence), "length" (max_new_tokens) or "cache" (the
max_cache_len guard).

generate(..., controls=...) and serve(..., controls=...) add a logit bias, banned token sequences ("bad words") and
min_tokens (LogitControls, one per request).  Like the penalties they depend on each draft row's own context - the
output so far plus the draft tokens on its path - and on the output position it predicts, so one
samd_apply_logit_controls launch rewrites every live row right after the penalties, and greedy verification stays
lossless against plain controlled greedy decoding.
"""
from __future__ import annotations

import dataclasses
import math
import numbers
from typing import Iterable, Iterator, List, Mapping, Optional, Sequence, Tuple, Union

import torch
from transformers.cache_utils import Cache, CacheLayerMixin

from . import _cabi as K
from . import engine as E

_cabi = K                       # (BatchedSamOnlyDecoder takes a parameter named K)


@dataclasses.dataclass(frozen=True)
class SamplingParams:
    """Sampled decoding of one request (the fields of the reference's SamdGenerationConfig with greedy=False, plus the
    seed of the request's device Philox stream).  temperature >= 1e-5 (unless greedy), 0 <= top_p <= 1 (active below 1,
    0 = off), top_k >= 0 (0 = off), 0 <= seed < 2**63.  greedy=True decodes this request greedily inside a sampled call:
    its tokens are plain greedy decoding and it makes no draw.  The decoders check the values of every request when it is
    pulled and name its index in the error."""
    temperature: float = 1.0
    top_p: float = 0.0
    top_k: int = 0
    seed: int = 0
    greedy: bool = False

    def problem(self) -> Optional[str]:
        """What is wrong with these values (None: nothing)."""
        if not isinstance(self.greedy, bool):
            return f"greedy must be a bool, got {self.greedy!r}"
        if not self.greedy and not self.temperature >= 1e-5:
            return f"temperature must be >= 1e-5, got {self.temperature}"
        if not 0.0 <= self.top_p <= 1.0:
            return f"top_p must be in [0, 1], got {self.top_p}"
        if not isinstance(self.top_k, int) or self.top_k < 0:
            return f"top_k must be an int >= 0, got {self.top_k!r}"
        if not isinstance(self.seed, int) or not 0 <= self.seed < 2 ** 63:
            return f"seed must be an int in [0, 2**63), got {self.seed!r}"
        return None


@dataclasses.dataclass(frozen=True)
class Penalties:
    """Penalties on repeated tokens for one request, applied to the logits before temperature, top-p and top-k (the
    order of HF and vLLM).  repetition_penalty r > 0 (HF's RepetitionPenaltyLogitsProcessor: every token of the prompt
    or the output so far is divided by r, or multiplied by r when negative); presence_penalty p and frequency_penalty f
    in [-2, 2] (the OpenAI API: p is subtracted once from a token that occurs in the output, f once per occurrence; the
    prompt is not counted).  The defaults change nothing.  The decoders check the values of every request when it is
    pulled and name its index in the error."""
    repetition_penalty: float = 1.0
    presence_penalty: float = 0.0
    frequency_penalty: float = 0.0

    def problem(self) -> Optional[str]:
        """What is wrong with these values (None: nothing)."""
        for name in ("repetition_penalty", "presence_penalty", "frequency_penalty"):
            v = getattr(self, name)
            if isinstance(v, bool) or not isinstance(v, (int, float)) or not math.isfinite(v):
                return f"{name} must be a finite float, got {v!r}"
        if not self.repetition_penalty > 0:
            return f"repetition_penalty must be > 0, got {self.repetition_penalty!r}"
        for name in ("presence_penalty", "frequency_penalty"):
            if not -2.0 <= getattr(self, name) <= 2.0:
                return f"{name} must be in [-2, 2], got {getattr(self, name)!r}"
        return None


@dataclasses.dataclass(frozen=True)
class StopSequences:
    """Stop sequences of one request: at most 16 sequences of 1 to 16 token ids in [0, V) each (ids, not strings: a
    string that tokenizes several ways is passed as one sequence per tokenization).  The request's output ends at the
    earliest output position where one of them ends - matched against the output alone, never the prompt - and the
    matched tokens stay in it, as EOS does; among sequences ending there the lowest index wins.  StopSequences(()) stops
    nothing.  The decoders check the sequences of every request when it is pulled and name its index in the error."""
    sequences: Sequence[Sequence[int]] = ()

    def problem(self, vocab: int) -> Optional[str]:
        """What is wrong with these sequences for a vocabulary of `vocab` tokens (None: nothing)."""
        return _sequences_problem(self.sequences, vocab, "sequences", "sequence", K.STOP_MAX_SEQS, K.STOP_MAX_LEN)


def _sequences_problem(seqs, vocab: int, field: str, item: str, max_seqs: int, max_len: int) -> Optional[str]:
    """What is wrong with a list of token id sequences `seqs` (the field `field`, whose entries are called `item`): at
    most max_seqs sequences of 1 to max_len ids in [0, vocab) each (None: nothing)."""
    if not isinstance(seqs, (list, tuple)):
        return f"{field} must be a list or tuple of token id sequences, got {type(seqs).__name__}"
    if len(seqs) > max_seqs:
        return f"at most {max_seqs} {item}s, got {len(seqs)}"
    for j, seq in enumerate(seqs):
        if not isinstance(seq, (list, tuple)):
            return f"{item} {j} must be a list or tuple of token ids, got {type(seq).__name__}"
        if not 1 <= len(seq) <= max_len:
            return f"{item} {j} must have 1 to {max_len} token ids, got {len(seq)}"
        for t in seq:
            if isinstance(t, bool) or not isinstance(t, numbers.Integral) or not 0 <= t < vocab:
                return f"{item} {j}: token ids must be ints in [0, {vocab}), got {t!r}"
    return None


@dataclasses.dataclass(frozen=True)
class LogitControls:
    """Logit controls of one request, applied to every logits row after the penalties and before temperature, top-p and
    top-k.  The decoders check the values of every request when it is pulled and name its index in the error.

    logit_bias: {token_id: bias} or a sequence of (token_id, bias) pairs (a repeated id is an error), at most 256
    distinct ids in [0, V).  A bias is a float in [-100, 100] (the OpenAI range), added to the logit in fp32 and rounded
    once into the logits' dtype, or -inf: the token is banned.
    bad_words: at most 16 sequences of 1 to 16 token ids.  Where the request's context - its output so far, never the
    prompt, then the tokens a draft row's path adds - ends with a sequence's first L - 1 ids, its last id is banned (a
    one-id sequence is banned everywhere), so the output never contains a bad word.
    min_tokens: an int m in [0, max_new_tokens].  While fewer than m tokens have been emitted, the decoder's
    eos_token_id and the last id of every stop sequence (stop=) whose head ends the context are banned, so neither EOS
    nor a stop sequence ends the request before m tokens (HF's MinNewTokensLengthLogitsProcessor, extended to
    multi-token stops); the max_cache_len guard still may.
    A banned token's logit is -inf.  LogitControls() changes nothing."""
    logit_bias: Union[Mapping[int, float], Sequence[Tuple[int, float]]] = ()
    bad_words: Sequence[Sequence[int]] = ()
    min_tokens: int = 0

    def bias_items(self) -> list:
        """logit_bias as a list of (token_id, bias) pairs."""
        lb = self.logit_bias
        return list(lb.items()) if isinstance(lb, Mapping) else list(lb)

    def problem(self, vocab: int) -> Optional[str]:
        """What is wrong with these values for a vocabulary of `vocab` tokens (None: nothing)."""
        lb = self.logit_bias
        if not isinstance(lb, (Mapping, list, tuple)):
            return f"logit_bias must be a mapping or a sequence of (token_id, bias) pairs, got {type(lb).__name__}"
        seen = set()
        for k, pair in enumerate(self.bias_items()):
            if not isinstance(pair, (list, tuple)) or len(pair) != 2:
                return f"logit_bias entry {k} must be a (token_id, bias) pair, got {pair!r}"
            t, v = pair
            if isinstance(t, bool) or not isinstance(t, numbers.Integral) or not 0 <= t < vocab:
                return f"logit_bias: token ids must be ints in [0, {vocab}), got {t!r}"
            if int(t) in seen:
                return f"logit_bias: token id {int(t)} appears more than once"
            seen.add(int(t))
            if isinstance(v, bool) or not isinstance(v, numbers.Real) or not (-100.0 <= v <= 100.0 or v == -math.inf):
                return f"logit_bias: the bias of token {int(t)} must be a float in [-100, 100] or -inf, got {v!r}"
        if len(seen) > K.BIAS_MAX:
            return f"logit_bias: at most {K.BIAS_MAX} token ids, got {len(seen)}"
        bad = _sequences_problem(self.bad_words, vocab, "bad_words", "bad word", K.BAD_MAX_SEQS, K.BAD_MAX_LEN)
        if bad:
            return bad
        m = self.min_tokens
        if isinstance(m, bool) or not isinstance(m, numbers.Integral) or m < 0:
            return f"min_tokens must be an int >= 0, got {m!r}"
        return None


def _check_logprobs(logprobs) -> Optional[int]:
    """generate() / serve()'s `logprobs`: None, or the number of alternatives per token, an int in [0, 8]."""
    if logprobs is not None and (isinstance(logprobs, bool) or not isinstance(logprobs, int) or not 0 <= logprobs <= 8):
        raise K.SamdError(f"logprobs must be None or an int in [0, 8], got {logprobs!r}")
    return logprobs


def _logprob_lists(rows: torch.Tensor, n: int) -> tuple:
    """One finished request's host rows [L, 1 + 2n] (log-probability | top-n values | top-n ids) as serve() returns them:
    (logprobs, top_logprobs as n (token_id, logprob) pairs per token, or None for n = 0)."""
    top = [list(zip(i, v)) for i, v in zip(rows[:, 1 + n:].long().tolist(), rows[:, 1:1 + n].tolist())] if n else None
    return rows[:, 0].tolist(), top


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

    def begin(self, n_new: int, kv_len: int, slots: Optional[torch.Tensor] = None, base: Optional[torch.Tensor] = None):
        """Set up the next forward.  By default it carries every request and writes its new rows at cache_len[b] + t.
        With `slots` (int64 [n]) it carries only those requests, in that order - a prefill of newly admitted requests:
        rows 0 .. n_new - 1 of those slots are written and attention reads those slots alone; with `base` (int32 [n])
        too, rows base[i] .. base[i] + n_new - 1 of slot i (the suffix of a prompt whose first base[i] rows are there)."""
        ar = torch.arange(n_new, device=self.kv.device)[None, :]
        if slots is None:
            # (clamped: a finished request still rides along in the batch; its rows may be written past its end, never
            # past the cache)
            self._slots = None
            self.rows = (self.cache_len.long()[:, None] + ar).clamp_(max=self.max_len - 1)
        else:
            self._slots = slots[:, None]
            if base is None:
                self.rows = ar.expand(slots.numel(), -1)
            else:                       # (a right-padded suffix's pad rows likewise: clamped, never past the cache)
                self.rows = (base.long()[:, None] + ar).clamp_(max=self.max_len - 1)
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

    def kv_table(self) -> tuple:
        """The 2L tensors as the C ABI sees them (engine.kv_table), built once."""
        if getattr(self, "_kv_table", None) is None:
            self._kv_table = E.kv_table([self.kv[i] for i in range(self.kv.shape[0])], self.kv.device)
        return self._kv_table


class BatchedSamdDecoder:
    """Batched lossless speculative decoding with the samd flavour: B slots, generate() for exactly B prompts in
    lockstep, serve() for any number of requests (continuous batching).

    Prefix reuse (max_prefixes > 0): add_prefix(tokens) registers a prompt head - a system prompt, a few-shot block, a
    document, an earlier chat turn - once, in a pool of max_prefixes entries: its KV rows (a RaggedKVCache of
    max_prefixes rows), its automaton and static cursor (a DynSamBatch and DraftEngine of max_prefixes requests), its
    greedy next token and, in Token-Recycle tree mode, the top-8 rows of its positions.  Every admission, in serve() and
    generate(), then starts a request whose prompt begins with a registered prefix P (the longest such P; a prompt equal
    to P included) from copies of that state - samd_kv_copy_rows for rows [0, len(P)), samd_dyn_clone for the automaton
    - and runs only the rest of the prompt through the LM and the step kernel.  The outputs are the same as without the
    pool.  With max_prefixes = 0 (the default) nothing is allocated and add_prefix raises."""

    def __init__(self, lm, batch: int, max_cache_len: int, n_predicts: int = 16, len_bias: int = 5, len_threshold: int = 5,
                 static: Optional[E.StaticSamDevice] = None, eos_token_id: Optional[int] = None, max_tokens: int = 16384,
                 dtype=torch.float16, device="cuda", tree: Optional[List[List[int]]] = None, max_prefixes: int = 0):
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
        self._init_pool(max_prefixes)

    def _init_pool(self, max_prefixes: int):
        """The prefix pool (nothing at all when max_prefixes is 0)."""
        self._prefixes = self.pool = None
        if max_prefixes > 0:
            cache = RaggedKVCache(self.lm.config, max_prefixes, self.cache.max_len, self.dtype, self.device)
            dyn = E.DynSamBatch(max_prefixes, self.dyn.max_tokens, self.device)
            # ingestion only (no lookup); it has cursors on the decoder's static automaton
            eng = E.DraftEngine(dyn, self.eng.static, self.eng.flavour, n_predicts=self.eng.n_predicts)
            self.pool = dict(cache=cache, dyn=dyn, eng=eng)
            self._prefixes = [None] * max_prefixes      # per pool row: dict(tokens, ids, last, topk) or None
            self._slot_plen = [0] * self.B

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
                         attention_mask=mask[:, None]).logits.contiguous()
        if not self.ver_bound:
            self.ver.bind_kv([self.cache.kv[i] for i in range(self.cache.kv.shape[0])])
            self.ver_bound = True
        n_nodes, ret = self._n_nodes[kind].contiguous(), self._ret[kind].contiguous()
        n_paths = self._n_paths[kind].contiguous()
        self._penalize(logits, draft, ret, n_nodes, n_paths)
        self._control(logits, draft, ret, n_nodes, n_paths)
        return self.ver.verify(logits, draft, ret, cache_len=self.cache.cache_len, move_kv=True, n_nodes=n_nodes,
                               n_paths=n_paths, out=res, recycle=self.table), logits, n_nodes

    def _draft_forward_verify(self, kv_len: int) -> tuple:
        """Drafts in, LM forward, fused verify: the part of a step that depends on the draft flavour.  Returns the verify
        outputs, the logits they were computed from and every request's live row count (None: all T rows)."""
        st, T, cache = self._st, self.T, self.cache
        self.eng.step(st["acc_tokens"], st["acc_count"], st["start"])              # update(accepted) + lookup(start): one launch
        cache.begin(T, kv_len)
        if self.tree is not None:
            return self._tree_step(st["start"], kv_len, st["res"])
        draft = self.eng.draft
        draft[:, 0] = st["start"]                                                  # short matches verify the start token only
        pos = cache.cache_len.long()[:, None] + self._ar[None, :]
        logits = self.lm(input_ids=draft.long(), position_ids=pos, past_key_values=cache,
                         attention_mask=self._mask(T, kv_len, cache.cache_len)).logits.contiguous()
        self._penalize(logits, draft)
        self._control(logits, draft)
        if self._sampled:                                      # identity path: no row moves, the commit sets cache_len
            return self._verify_sample(logits, draft, None), logits, None
        return self.ver.verify(logits, draft, None, cache_len=cache.cache_len, out=st["res"]), logits, None

    def _penalize(self, logits: torch.Tensor, tokens: torch.Tensor, retrieve: Optional[torch.Tensor] = None,
                  n_nodes: Optional[torch.Tensor] = None, n_paths: Optional[torch.Tensor] = None):
        """Between the LM forward and the verify launch of a penalized call: every live draft row penalized in place from
        its own path (identity chain without `retrieve`), one samd_apply_penalties launch.  Nothing otherwise."""
        if self._penalized:
            st = self._st
            E.apply_penalties(logits, st["pen_counts"], st["pen_r"], st["pen_p"], st["pen_f"], tokens=tokens,
                              retrieve=retrieve, n_nodes=n_nodes, n_paths=n_paths, done=st["done"])

    def _control(self, logits: torch.Tensor, tokens: torch.Tensor, retrieve: Optional[torch.Tensor] = None,
                 n_nodes: Optional[torch.Tensor] = None, n_paths: Optional[torch.Tensor] = None):
        """Right after _penalize, in a call with logit controls: every live draft row's bias, bad words and min_tokens
        bans from its own context (the slot's output so far, then its path) and the output position it predicts, one
        samd_apply_logit_controls launch.  Nothing otherwise."""
        if self._controlled:
            st = self._st
            stops = dict(stop_tokens=st["stop_tok"], stop_len=st["stop_len"]) if self._stopped else {}
            E.apply_logit_controls(logits, st["ctl_bias_ids"], st["ctl_bias"], st["ctl_bias_n"], st["ctl_bad_tok"],
                                   st["ctl_bad_len"], st["ctl_min"], tokens=tokens, retrieve=retrieve, n_nodes=n_nodes,
                                   n_paths=n_paths, done=st["done"], hist=st["out"], hist_len=st["out_len"],
                                   eos=None if self.eos is None else int(self.eos), **stops)

    def _verify_sample(self, logits: torch.Tensor, tokens: torch.Tensor, retrieve: Optional[torch.Tensor], **kw) -> dict:
        """samd_verify_sample_requests with every slot's processor, greedy flag and Philox stream; finished slots make no
        draw and accept nothing."""
        st = self._st
        return self.ver.verify_sample(logits, tokens, retrieve, st["temperature"], st["top_p"], st["top_k"], st["seed"],
                                      st["offset"], greedy=st["greedy"], done=st["done"], out=st["res"], **kw)

    # ---- one decode step, entirely on the device (no host read anywhere: it is what gets captured in a CUDA graph) ----
    def _step_body(self, kv_len: int):
        st, T = self._st, self.T
        cache = self.cache
        # a request whose step could run past the cache is finished (samd_model.py:251-254)
        st["done"].logical_or_(cache.cache_len + T > cache.max_len)
        saved_len = cache.cache_len.clone()
        res, logits, n_nodes = self._draft_forward_verify(kv_len)
        st["res"] = res
        lp = None
        if self._logprobs is not None:                     # the accepted rows' log-probabilities: one more launch
            n = self._logprobs
            lp = self._lp_res[n] = self.ver.token_logprobs(logits, res["indices"], res["accept_len"], res["tokens"],
                                                           res["next_token"], n_top=n, n_nodes=n_nodes, done=st["done"],
                                                           out=self._lp_res.get(n))
        self._commit(res, saved_len, lp)

    def _commit(self, res: dict, saved_len: torch.Tensor, lp: Optional[dict] = None):
        """EOS truncation, the stop-sequence cut (calls with stops), emission up to each slot's own limit, cache lengths, the next step's inputs, history and the
        host flag.  With `lp` (token_logprobs of this step) the emitted tokens' log-probabilities go to the columns of
        st["lp"] (and top-n lists to st["lp_ids"] / st["lp_top"]) parallel to st["out"]: emitted token 0 is the start
        token, predicted by the previous step's last row (st["start_lp"]), token k >= 1 is scored position k - 1."""
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
        if self._stopped:                  # the earliest stop sequence among the tokens the step would emit: cut there
            cand = torch.minimum(n_acc, room)
            cut, hit = E.match_stops(res["tokens"], cand, st["out"], st["out_len"], st["stop_tok"], st["stop_len"],
                                     out_count=cand, out_hit=st["stop_step"])
            stopped = hit >= 0
            n_acc = torch.where(stopped, cut, n_acc)
            done.logical_or_(stopped)
            torch.maximum(st["stop_hit"], hit, out=st["stop_hit"])            # (-1 from admission until a hit)
        n_emit = torch.minimum(n_acc, room)
        out = st["out"]
        cols = st["out_len"].long()[:, None] + ar[None, :]
        keep = ar[None, :] < n_emit[:, None]
        cols = torch.where(keep, cols, torch.full_like(cols, out.shape[1] - 1))
        emitted = torch.where(keep, res["tokens"], torch.zeros_like(res["tokens"]))
        out.scatter_(1, cols, emitted)
        if self._penalized:                                                        # the emitted tokens join the slot's counts
            st["pen_counts"].scatter_add_(1, emitted.long(), keep.int())
        if lp is not None:
            self._commit_logprobs(lp, cols, keep)
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

    def _commit_logprobs(self, lp: dict, cols: torch.Tensor, keep: torch.Tensor):
        """_commit's emission of the log-probabilities (and top-n lists) into the columns `cols` where `keep`, then the
        carry of the next start token's."""
        st, n, W = self._st, self._logprobs, cols.shape[1]
        step = torch.cat((st["start_lp"][:, None], lp["logprob"][:, :W - 1]), 1)
        st["lp"].scatter_(1, cols, torch.where(keep, step, torch.zeros_like(step)))
        st["start_lp"].copy_(lp["next_logprob"])
        if n:
            c, k = cols[:, :, None].expand(-1, -1, n), keep[:, :, None]
            for dst, start, top, nxt in (("lp_ids", "start_ids", "top_ids", "next_top_ids"),
                                         ("lp_top", "start_top", "top_logprob", "next_top_logprob")):
                step = torch.cat((st[start][:, None, :n], lp[top][:, :W - 1]), 1)
                st[dst][:, :, :n].scatter_(1, c, torch.where(k, step, torch.zeros_like(step)))
                st[start][:, :n].copy_(lp[nxt])

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
    def _init_state(self, max_limit: int, logprobs: bool = False, penalized: bool = False, stopped: bool = False,
                    controlled: bool = False):
        """Zeroed step state for requests of at most `max_limit` new tokens.  The tensors persist across calls (the
        captured graphs refer to them, and limits are per slot); they are reallocated, and the graphs dropped, only when
        a call needs longer outputs than any before.  The log-probability state is added by the first call that asks
        for log-probabilities, the penalty state by the first call with penalties, the stop state by the first call with
        stop sequences, the logit-control state by the first call with controls."""
        B, T, dev = self.B, self.T, self.device
        width = T if self.tree is None else self._ret.shape[2]
        cap = getattr(self, "_st_cap", None)
        if cap is None or cap < max_limit:
            mk = lambda *sh: torch.zeros(*sh, dtype=torch.int32, device=dev)
            # out: a slot's tokens plus spare columns; hist: its live steps (each emits >= 1 token, so at most max_limit)
            # plus a spare column; hlen: its live-step count; limit: its max_new_tokens
            # temperature .. offset: every slot's sampling parameters and the position of its Philox stream
            self._st = dict(start=mk(B), acc_tokens=mk(B, width), acc_count=mk(B), out=mk(B, max_limit + T), out_len=mk(B),
                            limit=mk(B), done=torch.zeros(B, dtype=torch.bool, device=dev), hist=mk(B, max_limit + 1),
                            hlen=mk(B), flag=mk(2 * B + 1), temperature=torch.ones(B, device=dev), top_p=torch.zeros(B, device=dev),
                            top_k=mk(B), greedy=torch.zeros(B, dtype=torch.uint8, device=dev),
                            seed=torch.zeros(B, dtype=torch.long, device=dev), offset=torch.zeros(B, dtype=torch.long, device=dev),
                            res=None, **self._extra_state(mk))
            self._st_cap, self._graphs, self._lp_res = max_limit, {}, {}
        else:
            for k, v in self._st.items():
                if k != "res":
                    v.zero_()
        if logprobs and "lp" not in self._st:
            # lp / lp_top / lp_ids: parallel to out (top-n lists at their widest, 8, so that a call with any n reuses
            # them); start_*: those of each slot's start token, carried from the step that predicted it
            W, f32 = self._st["out"].shape[1], lambda *sh: torch.zeros(*sh, device=dev)
            i32 = lambda *sh: torch.zeros(*sh, dtype=torch.int32, device=dev)
            self._st.update(lp=f32(B, W), lp_top=f32(B, W, 8), lp_ids=i32(B, W, 8), start_lp=f32(B), start_top=f32(B, 8),
                            start_ids=i32(B, 8))
        if penalized and "pen_counts" not in self._st:
            # pen_counts: every slot's output count per token, E.PENALTY_PROMPT_BIT set for its prompt's tokens;
            # pen_r / pen_p / pen_f: its repetition, presence and frequency penalties
            V = self.lm.config.vocab_size
            self._st.update(pen_counts=torch.zeros(B, V, dtype=torch.int32, device=dev), pen_r=torch.ones(B, device=dev),
                            pen_p=torch.zeros(B, device=dev), pen_f=torch.zeros(B, device=dev))
        if stopped and "stop_tok" not in self._st:
            # stop_tok / stop_len: every slot's stop sequences (length 0: unused); stop_hit: the index of the one that
            # ended it, -1 until then; stop_step: the step's match
            S, L = K.STOP_MAX_SEQS, K.STOP_MAX_LEN
            i32 = lambda *sh: torch.zeros(*sh, dtype=torch.int32, device=dev)
            self._st.update(stop_tok=i32(B, S, L), stop_len=i32(B, S), stop_hit=i32(B), stop_step=i32(B))
        if controlled and "ctl_min" not in self._st:
            # ctl_bias_ids / ctl_bias / ctl_bias_n: every slot's logit bias entries; ctl_bad_tok / ctl_bad_len: its bad
            # words (length 0: unused); ctl_min: its min_tokens
            M, S, L = K.BIAS_MAX, K.BAD_MAX_SEQS, K.BAD_MAX_LEN
            i32 = lambda *sh: torch.zeros(*sh, dtype=torch.int32, device=dev)
            self._st.update(ctl_bias_ids=i32(B, M), ctl_bias=torch.zeros(B, M, device=dev), ctl_bias_n=i32(B),
                            ctl_bad_tok=i32(B, S, L), ctl_bad_len=i32(B, S), ctl_min=i32(B))

    def _advance(self, kv_len: int, graph: bool) -> bool:
        """One decode step at key length `kv_len`: the bucket's CUDA graph, captured first if it is new, or the same body
        eagerly (one graph per bucket, greedy / sampled body, logprobs setting, penalized or not, stopped or not and
        controlled or not).  Returns `graph`,
        False from then on when the LM's forward cannot be captured."""
        if graph:
            B, dev, graphs = self.B, self.device, self._graphs
            key = (kv_len, self._sampled, self._logprobs, self._penalized, self._stopped, self._controlled)
            if key not in graphs:
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
                    graphs[key] = g
                    self.last_graphed = True
                except Exception:                          # an LM whose forward cannot be captured: same body, eagerly
                    graph = False
                    torch.cuda.synchronize(dev)
                restore()                                  # (capture does not run the work; the warm-up did)
                snap_dyn.close()
            if graph:
                graphs[key].replay()
                self.last_graphed = True
                return True
        self._step_body(kv_len)
        return False

    # ---- prefix reuse: a pool of registered prompt heads --------------------------------------------------------------
    @torch.inference_mode()
    def add_prefix(self, tokens: Sequence[int]) -> int:
        """Register a prompt head; returns its id (the id it already has when these tokens are registered).  The
        prefix's LM prefill runs alone into a pool row, its automaton and static cursor ingest it, and its greedy next
        token (and, in tree mode, the top-8 rows of its positions) are kept.  No slot and no captured graph is touched:
        it may be called between calls and while a serve() generator is suspended.  The logits row after the prefix is
        kept too: a prompt equal to the prefix starts from its argmax, or from a draw from its softmax when sampled."""
        tokens = tuple(int(t) for t in tokens)
        pid = self._check_prefix(tokens)
        if self._prefixes[pid] is not None:
            return pid
        pool, dev, n = self.pool, self.device, len(tokens)
        ids = torch.tensor([tokens], dtype=torch.long, device=dev)
        slot = torch.tensor([pid], dtype=torch.long, device=dev)
        logits = self._prefill_slots(ids, slot, cache=pool["cache"])
        P = pool["dyn"].n_requests
        eng = pool["eng"]
        eng.reset(torch.zeros(P, dtype=torch.uint8, device=dev).index_fill_(0, slot, 1))
        tok = torch.zeros(P, n, dtype=torch.int32, device=dev).index_copy_(0, slot, ids.to(torch.int32))
        eng.step(tok, torch.zeros(P, dtype=torch.int32, device=dev).index_fill_(0, slot, n), None)
        topk = self.table.topk(ids[0], logits[0]) if self.tree is not None else None
        self._prefixes[pid] = dict(tokens=tokens, ids=ids[0], last=logits[0, n - 1].clone(), topk=topk)
        return pid

    def drop_prefix(self, pid: int):
        """Forget prefix `pid`: no admission matches it any more and its pool row is free."""
        if self._prefixes is None or not 0 <= pid < len(self._prefixes) or self._prefixes[pid] is None:
            raise K.SamdError(f"drop_prefix: no registered prefix {pid}")
        self._prefixes[pid] = None

    def _check_prefix(self, tokens: tuple) -> int:
        """add_prefix's validation: the id of these tokens, or of the free pool row they would take."""
        if getattr(self, "_prefixes", None) is None:
            raise K.SamdError("add_prefix: this decoder has no prefix pool (construct it with max_prefixes > 0)")
        n, T, max_len, cap = len(tokens), self.T, self.cache.max_len, self.dyn.max_tokens
        if n == 0:
            raise K.SamdError("add_prefix: empty prefix")
        if n + T > max_len:
            raise K.SamdError(f"add_prefix: prefix of {n} tokens + one decode step of {T} does not fit "
                              f"max_cache_len={max_len}")
        if n + 1 + T > cap:
            raise K.SamdError(f"add_prefix: prefix of {n} tokens + one new token + one step exceeds the automaton "
                              f"capacity max_tokens={cap}")
        free = None
        for pid, e in enumerate(self._prefixes):
            if e is None:
                free = pid if free is None else free
            elif e["tokens"] == tokens:
                return pid
        if free is None:
            raise K.SamdError(f"add_prefix: the prefix pool is full ({len(self._prefixes)} prefixes); drop_prefix one first")
        return free

    def _longest_prefix(self, prompt: Sequence[int]) -> tuple:
        """(id, length) of the longest registered prefix P with prompt[:len(P)] == P, or (None, 0)."""
        best, best_len = None, 0
        for pid, e in enumerate(self._prefixes):
            if e is None:
                continue
            P = e["tokens"]
            n = len(P)
            if best_len < n <= len(prompt) and prompt[n - 1] == P[-1] and prompt[0] == P[0] and tuple(prompt[:n]) == P:
                best, best_len = pid, n
        return best, best_len

    # ---- admission: new requests into free slots, between two steps ---------------------------------------------------
    def _admit(self, reqs: List[tuple]) -> int:
        """Start the requests `reqs` = [(slot, prompt, limit, SamplingParams or None, Penalties or None, StopSequences or
        None, LogitControls or None)] in their (free) slots; returns the longest prompt.  Only the persistent state is written, in place, so the captured graphs stay valid."""
        dev = self.device
        n_max = max(len(r[1]) for r in reqs)
        if self._prefixes is not None:
            hits = [self._longest_prefix(r[1]) for r in reqs]
            for (b, *_), (_, n) in zip(reqs, hits):
                self._slot_plen[b] = n
            if any(pid is not None for pid, _ in hits):
                self._admit_prefixed(reqs, hits)
                return n_max
        ids = torch.zeros(len(reqs), n_max, dtype=torch.long)
        for i, (_, p, *_) in enumerate(reqs):
            ids[i, :len(p)] = torch.as_tensor(p, dtype=torch.long)
        meta = torch.tensor([[r[0] for r in reqs], [len(r[1]) for r in reqs], [r[2] for r in reqs]], dtype=torch.long)
        ids, meta = ids.to(dev), meta.to(dev)
        slots, lens, limits = meta[0], meta[1].to(torch.int32), meta[2].to(torch.int32)
        logits = self._prefill_slots(ids, slots)
        self._ingest(ids, slots, lens, logits)
        self._set_slots(slots, lens, limits, logits[torch.arange(slots.numel(), device=dev), lens.long() - 1], reqs)
        return n_max

    def _admit_prefixed(self, reqs: List[tuple], hits: List[tuple]):
        """_admit when some requests start with a registered prefix (pool row hits[i][0], length hits[i][1]; (None, 0)
        for the others): their KV rows [0, len(P)) come from the pool (one samd_kv_copy_rows launch), one LM forward
        runs over the suffixes alone (right padded, rows from len(P) on), the unmatched slots' drafters are reset and
        the matched ones cloned from the pool (one samd_dyn_clone launch, static-cursor rows copied), and one samd_step
        ingests the suffixes - count 0 for a prompt equal to its prefix, which starts from the logits row kept after the
        prefix."""
        dev, pool = self.device, self.pool
        n = len(reqs)
        sufs = [r[1][m:] for r, (_, m) in zip(reqs, hits)]
        n_suf = max(len(x) for x in sufs)
        hit = [i for i in range(n) if hits[i][0] is not None]
        fw = [i for i in range(n) if len(sufs[i])]                                   # requests with a suffix
        ids = torch.zeros(n, n_suf, dtype=torch.long)
        for i, x in enumerate(sufs):
            ids[i, :len(x)] = torch.as_tensor(x, dtype=torch.long)
        meta = torch.tensor([[r[0] for r in reqs], [len(r[1]) for r in reqs], [r[2] for r in reqs], [m for _, m in hits],
                             [len(x) for x in sufs], [-1 if pid is None else pid for pid, _ in hits]], dtype=torch.long)
        ids, meta = ids.to(dev), meta.to(dev)
        slots, lens, limits = meta[0], meta[1].to(torch.int32), meta[2].to(torch.int32)
        base, suf_lens, pids = meta[3].to(torch.int32), meta[4].to(torch.int32), meta[5]
        h = torch.tensor(hit, dtype=torch.long, device=dev)
        h_slots, h_pids = slots[h], pids[h]
        self._copy_prefix_kv(h_slots, h_pids, base[h])
        logits = None
        if fw:
            f = torch.tensor(fw, dtype=torch.long, device=dev)
            logits = self._prefill_slots(ids[f], slots[f], base=base[f], kv_len=max(hits[i][1] + len(sufs[i]) for i in fw))
        self._clone_drafters(slots, pids, h_slots, h_pids)
        self._ingest_suffixes(ids, slots, suf_lens, [(hits[i][0], len(sufs[i])) for i in range(n)], fw, logits)
        self.prefix_hits += len(hit)
        self.prefix_tokens += sum(hits[i][1] for i in hit)
        # the first start token comes from the row after the last suffix token, or after the prefix itself
        rows = [self._prefixes[hits[i][0]]["last"] if not len(sufs[i]) else None for i in range(n)]
        if fw:
            last = logits[torch.arange(len(fw), device=dev), suf_lens[f].long() - 1]
            for k, i in enumerate(fw):
                rows[i] = last[k]
        self._set_slots(slots, lens, limits, torch.stack(rows), reqs)

    def _copy_prefix_kv(self, slots: torch.Tensor, pids: torch.Tensor, plens: torch.Tensor):
        """KV rows [0, plens[i]) of pool row pids[i] into slot slots[i]: one samd_kv_copy_rows launch."""
        E.kv_copy_rows(self.cache.kv_table(), self.pool["cache"].kv_table(), slots.to(torch.int32),
                       pids.to(torch.int32), plens.to(torch.int32))

    def _clone_drafters(self, slots: torch.Tensor, pids: torch.Tensor, h_slots: torch.Tensor, h_pids: torch.Tensor):
        """Masked DraftModel.reset of the unmatched slots; the matched ones take a copy of their prefix's automaton (one
        samd_dyn_clone launch) and static cursor."""
        B, dev, pool = self.B, self.device, self.pool
        miss = slots[pids < 0]
        if miss.numel():
            self.eng.reset(torch.zeros(B, dtype=torch.uint8, device=dev).index_fill_(0, miss, 1))
        self.dyn.clone_from(pool["dyn"], h_pids.to(torch.int32), h_slots.to(torch.int32))
        if self.eng.static_cursor is not None:
            self.eng.static_cursor.index_copy_(0, h_slots, pool["eng"].static_cursor.index_select(0, h_pids))

    def _ingest_suffixes(self, ids: torch.Tensor, slots: torch.Tensor, suf_lens: torch.Tensor, parts: List[tuple],
                         fw: List[int], logits: Optional[torch.Tensor]):
        """DraftModel.update(suffix) of every admitted request in one launch (count 0 for every other slot), then in
        tree mode the successor table as an uncached admission leaves it: per request in admission order, its prefix's
        stored rows then its suffix rows, the last writer of a token winning (RecycleTable.apply)."""
        B, dev = self.B, self.device
        if ids.shape[1]:
            tokens = torch.zeros(B, ids.shape[1], dtype=torch.int32, device=dev).index_copy_(0, slots, ids.to(torch.int32))
            counts = torch.zeros(B, dtype=torch.int32, device=dev).index_copy_(0, slots, suf_lens)
            self.eng.step(tokens, counts, None)
        if self.tree is None:
            return
        rows_s = None
        if fw:
            f = torch.tensor(fw, dtype=torch.long, device=dev)
            valid = torch.arange(ids.shape[1], device=dev)[None, :] < suf_lens[f][:, None]
            rows_s = self.table.topk(ids[f][valid], logits[valid])
        toks, rows, at = [], [], 0
        for i, (pid, m) in enumerate(parts):                                         # admission order
            if pid is not None:
                e = self._prefixes[pid]
                toks.append(e["ids"])
                rows.append(e["topk"])
            if m:
                toks.append(ids[i, :m])
                rows.append(rows_s[at:at + m])
                at += m
        self.table.apply(torch.cat(toks), torch.cat(rows))
        if not self.ver_bound:
            self.ver.bind_kv([self.cache.kv[i] for i in range(self.cache.kv.shape[0])])
            self.ver_bound = True

    def _prefill_slots(self, ids: torch.Tensor, slots: torch.Tensor, base: Optional[torch.Tensor] = None,
                       kv_len: Optional[int] = None, cache: Optional[RaggedKVCache] = None) -> torch.Tensor:
        """LM prefill of the admitted prompts alone ([n, n_max], right padded) into KV rows 0 .. n_max - 1 of their
        slots: the cost follows the admitted prompts, not the batch.  With `base` (int32 [n]), the prompts are suffixes
        whose first base[i] rows are in the cache: rows and positions start at base[i], attention spans kv_len keys.
        `cache`: another cache than the decoder's (the prefix pool)."""
        n, n_max = ids.shape
        cache = self.cache if cache is None else cache
        if base is None:
            kv_len, base0 = n_max, torch.zeros(n, dtype=torch.int32, device=self.device)
        else:
            base0 = base
        cache.begin(n_max, kv_len, slots=slots, base=base)
        pos = base0.long()[:, None] + torch.arange(n_max, device=self.device)[None, :]
        return self.lm(input_ids=ids, position_ids=pos, past_key_values=cache,
                       attention_mask=self._mask(n_max, kv_len, base0)).logits

    def _ingest(self, ids: torch.Tensor, slots: torch.Tensor, lens: torch.Tensor, logits: torch.Tensor):
        """The admitted requests' drafters: masked DraftModel.reset (automaton and static cursor), then
        DraftModel.update(prompt) in one launch with count 0 for every other request, then the prefill hook."""
        B, dev = self.B, self.device
        self.eng.reset(torch.zeros(B, dtype=torch.uint8, device=dev).index_fill_(0, slots, 1))
        tokens = torch.zeros(B, ids.shape[1], dtype=torch.int32, device=dev).index_copy_(0, slots, ids.to(torch.int32))
        counts = torch.zeros(B, dtype=torch.int32, device=dev).index_copy_(0, slots, lens)
        self.eng.step(tokens, counts, None)
        self._prefill_hook(ids, lens, logits)

    def _set_slots(self, slots: torch.Tensor, lens: torch.Tensor, limits: torch.Tensor, rows: torch.Tensor,
                   reqs: List[tuple]):
        """The admitted slots' step state: cache length, stop sequences (calls with stops), sampling parameters and a
        fresh Philox stream (sampled calls), penalty state (penalized calls), logit controls (controlled calls), first
        start token from `rows` [n, V] (the logits after each prompt, penalized from the prompt alone in a penalized
        call, then controlled as the row predicting output position 0 in a controlled one: argmax, or a draw from the
        softmax) and, with logprobs, its log-probability, limit, and zero emitted tokens / history."""
        st, params = self._st, [r[3] for r in reqs]
        self.cache.cache_len.index_copy_(0, slots, lens)
        if self._stopped:
            n, S, L = len(reqs), K.STOP_MAX_SEQS, K.STOP_MAX_LEN
            tab = [[0] * (S * L + S) for _ in reqs]                           # [stop_tok | stop_len] per request
            for row, r in zip(tab, reqs):
                for j, seq in enumerate(r[5].sequences):
                    row[j * L:j * L + len(seq)] = [int(t) for t in seq]
                    row[S * L + j] = len(seq)
            tab = torch.tensor(tab, dtype=torch.int32).to(self.device)
            st["stop_tok"].index_copy_(0, slots, tab[:, :S * L].reshape(n, S, L))
            st["stop_len"].index_copy_(0, slots, tab[:, S * L:].contiguous())
            st["stop_hit"].index_fill_(0, slots, -1)
        if self._penalized:
            rows = self._admit_penalties(slots, rows, reqs)
        if self._controlled:
            rows = self._admit_controls(slots, rows, reqs)
        if self._sampled:
            dev = self.device
            f = torch.tensor([[sp.temperature, sp.top_p] for sp in params], dtype=torch.float32).T.contiguous().to(dev)
            i = torch.tensor([[sp.top_k, int(sp.greedy), sp.seed] for sp in params], dtype=torch.long).T.contiguous().to(dev)
            st["temperature"].index_copy_(0, slots, f[0])
            st["top_p"].index_copy_(0, slots, f[1])
            st["top_k"].index_copy_(0, slots, i[0].to(torch.int32))
            st["greedy"].index_copy_(0, slots, i[1].to(torch.uint8))
            st["seed"].index_copy_(0, slots, i[2])
            st["offset"].index_fill_(0, slots, 0)
            # depth 1: the kernel's walk is empty and the token is drawn from the plain softmax of the row (samd/utils.py
            # :173-179 with nothing accepted), as the reference's torch.multinomial after the prefill; greedy: its argmax
            n, V = rows.shape
            offs = st["offset"][slots]
            res = self.ver.verify_sample(rows.contiguous().view(n, 1, V), torch.zeros(n, 1, dtype=torch.int32, device=dev),
                                         None, st["temperature"][slots], st["top_p"][slots], st["top_k"][slots],
                                         st["seed"][slots], offs, greedy=st["greedy"][slots])
            st["offset"].index_copy_(0, slots, offs)
            first = res["next_token"]
        else:
            first = rows.argmax(-1).to(torch.int32)
        if self._logprobs is not None:                     # the first token's log-probability, from the same row
            n, (m, V) = self._logprobs, rows.shape
            lp = self.ver.token_logprobs(rows.contiguous().view(m, 1, V), None,
                                         torch.ones(m, dtype=torch.int32, device=self.device), None, first, n_top=n)
            st["start_lp"].index_copy_(0, slots, lp["next_logprob"])
            if n:
                st["start_ids"][slots, :n] = lp["next_top_ids"]
                st["start_top"][slots, :n] = lp["next_top_logprob"]
        st["start"].index_copy_(0, slots, first)
        st["limit"].index_copy_(0, slots, limits)
        for k in ("acc_count", "out_len", "hlen"):
            st[k].index_fill_(0, slots, 0)
        st["done"].index_fill_(0, slots, False)

    def _admit_penalties(self, slots: torch.Tensor, rows: torch.Tensor, reqs: List[tuple]) -> torch.Tensor:
        """The admitted slots' penalty state - output counts zeroed, the whole prompt's tokens marked seen, r / p / f
        written - and a penalized copy of `rows` (the prefix pool's stored rows stay as they are)."""
        st, dev, V = self._st, self.device, rows.shape[-1]
        n, n_max = len(reqs), max(len(r[1]) for r in reqs)
        ids = torch.zeros(n, n_max, dtype=torch.long)
        for i, r in enumerate(reqs):
            ids[i, :len(r[1])] = torch.as_tensor(r[1], dtype=torch.long)
            ids[i, len(r[1]):] = r[1][0]                       # pads repeat a prompt token: token 0 is not marked
        vals = torch.tensor([[r[4].repetition_penalty, r[4].presence_penalty, r[4].frequency_penalty] for r in reqs],
                            dtype=torch.float32).T.contiguous()
        ids, vals = ids.to(dev), vals.to(dev)
        st["pen_counts"].index_copy_(0, slots, torch.zeros(n, V, dtype=torch.int32, device=dev).scatter_(
            1, ids, E.PENALTY_PROMPT_BIT))
        for k, name in enumerate(("pen_r", "pen_p", "pen_f")):
            st[name].index_copy_(0, slots, vals[k])
        rows = rows.clone()
        E.apply_penalties(rows.view(n, 1, V), st["pen_counts"], st["pen_r"], st["pen_p"], st["pen_f"],
                          slots=slots.to(torch.int32))
        return rows

    def _admit_controls(self, slots: torch.Tensor, rows: torch.Tensor, reqs: List[tuple]) -> torch.Tensor:
        """The admitted slots' logit-control tables, and a controlled copy of `rows`: each is the row predicting output
        position 0, with no context (the prefix pool's stored rows stay as they are)."""
        st, n, V = self._st, len(reqs), rows.shape[-1]
        M, S, L = K.BIAS_MAX, K.BAD_MAX_SEQS, K.BAD_MAX_LEN
        ids, bias = torch.zeros(n, M, dtype=torch.int32), torch.zeros(n, M)
        small = torch.zeros(n, 2 + S + S * L, dtype=torch.int32)                 # [bias_n | min | bad_len | bad_tok]
        for i, r in enumerate(reqs):
            lc = r[6]
            items = lc.bias_items()
            if items:
                ids[i, :len(items)] = torch.tensor([int(t) for t, _ in items], dtype=torch.int32)
                bias[i, :len(items)] = torch.tensor([float(v) for _, v in items], dtype=torch.float32)
            small[i, 0], small[i, 1] = len(items), int(lc.min_tokens)
            for j, seq in enumerate(lc.bad_words):
                small[i, 2 + j] = len(seq)
                small[i, 2 + S + j * L:2 + S + j * L + len(seq)] = torch.tensor([int(t) for t in seq], dtype=torch.int32)
        ids, bias, small = ids.to(self.device), bias.to(self.device), small.to(self.device)
        st["ctl_bias_ids"].index_copy_(0, slots, ids)
        st["ctl_bias"].index_copy_(0, slots, bias)
        st["ctl_bias_n"].index_copy_(0, slots, small[:, 0].contiguous())
        st["ctl_min"].index_copy_(0, slots, small[:, 1].contiguous())
        st["ctl_bad_len"].index_copy_(0, slots, small[:, 2:2 + S].contiguous())
        st["ctl_bad_tok"].index_copy_(0, slots, small[:, 2 + S:].reshape(n, S, L))
        stops = dict(stop_tokens=st["stop_tok"], stop_len=st["stop_len"]) if self._stopped else {}
        rows = rows.clone()
        E.apply_logit_controls(rows.view(n, 1, V), st["ctl_bias_ids"], st["ctl_bias"], st["ctl_bias_n"],
                               st["ctl_bad_tok"], st["ctl_bad_len"], st["ctl_min"], slots=slots.to(torch.int32),
                               eos=None if self.eos is None else int(self.eos), **stops)
        return rows

    # ---- the decode loop of generate() and serve() --------------------------------------------------------------------
    def _run(self, requests: Iterator[tuple], max_limit: int, graph: bool, check_every: int, sampled: bool = False,
             logprobs: Optional[int] = None, penalized: bool = False, stopped: bool = False, controlled: bool = False):
        """Decode the validated requests (index, prompt, limit, SamplingParams or None, Penalties or None, StopSequences
        or None, LogitControls or None) of `requests`, at most B at a time, with the greedy step body or (sampled) the
        sampled one; with `logprobs` (0 .. 8) the step also scores the accepted rows, `penalized` penalizes the draft
        rows before verification, `controlled` then applies each request's logit controls, and `stopped` cuts each
        request's output at its first stop sequence.  The decode step has no host synchronisation in it: it is captured once per key-length bucket (64
        positions) as a CUDA graph and replayed.  Once every `check_every` steps the host reads [done | out_len | longest cache] in one copy; it then
        yields (index, tokens, accept_lengths, slot, (logprobs, top_logprobs) or None, finish reason, stop index or None)
        for every request found finished (their rows and stop indices in one more copy, their log-probabilities in one
        more),
        admits queued requests into the free slots, and sizes the next steps' key length from the longest cache.  A
        finished request keeps its slot - riding along, emitting nothing - until that check.  Statistics go to
        self._run_stats."""
        B, T, dev = self.B, self.T, self.device
        self._init_state(max_limit, logprobs is not None, penalized, stopped, controlled)
        self._sampled, self._logprobs, self._penalized, self._stopped = sampled, logprobs, penalized, stopped
        self._controlled = controlled
        st = self._st
        run = self._run_id = getattr(self, "_run_id", 0) + 1
        self.eng.reset()
        self.cache.cache_len.zero_()
        st["done"].fill_(True)                                                     # an empty slot rides along finished
        owner = [None] * B                                                         # request index in each slot
        limit_of = [0] * B                                                         # and its max_new_tokens
        W, max_accept = st["out"].shape[1], st["acc_tokens"].shape[1]              # (the most one step adds to a cache)
        H = st["hist"].shape[1]
        flag_host = torch.zeros(2 * B + 1, dtype=torch.int32).pin_memory()
        steps = syncs = since = admissions = live_steps = 0
        self.prefix_hits = self.prefix_tokens = 0
        self.last_graphed = False

        def admit() -> int:
            nonlocal admissions
            reqs = []
            for b in range(B):
                if owner[b] is None:
                    r = next(requests, None)
                    if r is None:
                        break
                    owner[b], limit_of[b] = r[0], r[2]
                    reqs.append((b,) + tuple(r[1:]))
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
                cols = (st["out"][idx], st["hist"][idx], st["hlen"][idx, None])
                if stopped:
                    cols += (st["stop_hit"][idx, None],)
                rows = torch.cat(cols, 1).tolist()
                lps = [None] * len(fin)
                if logprobs is not None:                   # [f, W, 1 + 2n]: log-probability | top-n values | top-n ids
                    n = logprobs
                    lpr = torch.cat((st["lp"][idx, :, None], st["lp_top"][idx, :, :n], st["lp_ids"][idx, :, :n].float()),
                                    2).cpu()
                    lps = [_logprob_lists(lpr[k, :flag[B + b]], n) for k, b in enumerate(fin)]
                for b, r, lp in zip(fin, rows, lps):
                    i, owner[b] = owner[b], None
                    hist = r[W:W + r[W + H]]
                    live_steps += len(hist)
                    tokens, hit = r[:flag[B + b]], r[W + H + 1] if stopped else -1
                    yield i, tokens, hist, b, lp, self._finish_reason(tokens, hit, limit_of[b]), hit if hit >= 0 else None
                    if self._run_id != run:
                        raise K.SamdError("the decoder ran another generate() / serve() while this serve() was suspended")
            kv_hi = max(kv_hi, admit())
        self._run_stats = dict(steps_run=steps, host_syncs=syncs, graphed=self.last_graphed, graphs=len(self._graphs),
                               admissions=admissions, live_slot_steps=live_steps, **self._extra_stats())
        if self._prefixes is not None:
            self._run_stats.update(prefix_hits=self.prefix_hits, prefix_tokens=self.prefix_tokens)

    def _finish_reason(self, tokens: List[int], stop_hit: int, limit: int) -> str:
        """Why a finished request ended: "stop" (a stop sequence, or EOS - truncation keeps it as the last token),
        "length" (max_new_tokens) or "cache" (the max_cache_len guard, which finished it before either)."""
        if stop_hit >= 0 or (self.eos is not None and tokens and tokens[-1] == self.eos):
            return "stop"
        return "length" if len(tokens) >= limit else "cache"

    @torch.inference_mode()
    def generate(self, prompts: Sequence[Sequence[int]], max_new_tokens: int, graph: bool = True, check_every: int = 4,
                 sampling: Union[None, SamplingParams, Sequence[SamplingParams]] = None, logprobs: Optional[int] = None,
                 penalties: Union[None, Penalties, Sequence[Penalties]] = None,
                 stop: Union[None, StopSequences, Sequence[StopSequences]] = None,
                 controls: Union[None, LogitControls, Sequence[LogitControls]] = None):
        """Lossless batched speculative decoding of exactly B prompts in lockstep (request b in slot b), up to
        max_new_tokens each.  The host reads the finished flags once every `check_every` steps - 1 / check_every host
        syncs per step - so a finished batch may run up to check_every - 1 idle steps (every request done: nothing is
        emitted).  graph=False runs the same body eagerly.  Returns (tokens per request, stats); stats["accept_lengths"]
        holds every request's accepted tokens per step, padded with 0 to the longest request's `steps`.  `sampling`,
        `logprobs`, `penalties`, `stop` and `controls`: as in serve(); with logprobs, stats["logprobs"] (and, for logprobs > 0,
        stats["top_logprobs"]) hold every request's list.  stats["finish_reasons"] holds every request's finish reason
        and, with stop, stats["stop_indices"] its stop index."""
        logprobs = _check_logprobs(logprobs)
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
        V = self.lm.config.vocab_size
        reqs = self._with_sampling(((i, p, max_new_tokens) for i, p in enumerate(prompts)), sampling)
        reqs = self._with_controls(self._with_stops(self._with_penalties(reqs, penalties), stop, V), controls, V)
        out, acc, lps, why, hits = [None] * B, [None] * B, [None] * B, [None] * B, [None] * B
        for i, tokens, hist, _, lp, reason, hit in self._run(reqs, max_new_tokens, graph, check_every, sampling is not None,
                                                             logprobs, penalties is not None, stop is not None,
                                                             controls is not None):
            out[i], acc[i], lps[i], why[i], hits[i] = tokens, hist, lp, reason, hit
        n_live = max(len(a) for a in acc)
        s = self._run_stats
        stats = dict(steps=n_live, steps_run=s["steps_run"], host_syncs=s["host_syncs"], graphed=s["graphed"],
                     graphs=s["graphs"], accept_lengths=[a + [0] * (n_live - len(a)) for a in acc], finish_reasons=why,
                     **self._extra_stats())
        if stop is not None:
            stats["stop_indices"] = hits
        if logprobs is not None:
            stats["logprobs"] = [lp[0] for lp in lps]
            if logprobs:
                stats["top_logprobs"] = [lp[1] for lp in lps]
        return out, stats

    @torch.inference_mode()
    def serve(self, prompts: Iterable[Sequence[int]], max_new_tokens: Union[int, Sequence[int]], graph: bool = True,
              check_every: int = 4, sampling: Union[None, SamplingParams, Sequence[SamplingParams]] = None,
              logprobs: Optional[int] = None, penalties: Union[None, Penalties, Sequence[Penalties]] = None,
              stop: Union[None, StopSequences, Sequence[StopSequences]] = None,
              controls: Union[None, LogitControls, Sequence[LogitControls]] = None):
        """Continuous batching: decode any number of requests through the B slots, refilling a slot with the next queued
        request as soon as the host sees its request finished (once every `check_every` steps).  `prompts` is consumed
        lazily and in order; `max_new_tokens` is one limit for all or a sequence with one per request.  Yields
        (index, tokens, {"slot", "accept_lengths", "finish_reason"}) per request in completion order; `tokens` are what generate() emits
        for that prompt, `accept_lengths` has one entry per live decode step.  A request is validated when it is pulled
        (SamdError naming its index).  self.serve_stats is set once the generator is exhausted: steps_run, host_syncs
        (flag reads), graphed, graphs, admissions, live_slot_steps (slot-steps of unfinished requests) and, for
        BatchedSamOnlyDecoder, tree_steps.  One call at a time: a generate() or serve() call while this generator is
        suspended ends it (it raises when resumed); an abandoned generator leaves the decoder usable.

        With a prefix pool (max_prefixes > 0) every request starts from the longest registered prefix its prompt begins
        with (add_prefix may be called while this generator is suspended; it counts from the next admission on): its
        info also holds "prefix_len" (0 without a match), and serve_stats "prefix_hits" (requests that started from a
        prefix) and "prefix_tokens" (prompt tokens whose prefill and ingestion were skipped).

        `sampling` (None: greedy, lossless): one SamplingParams for every request - request i then uses the Philox key
        seed + i - or a sequence with one per request.  Each request's processor and stream are its own, so its tokens
        depend only on its prompt, parameters and seed; a request with greedy=True decodes greedily.  Not with
        Token-Recycle tree mode (tree=): SamdError.

        `logprobs` (None: none): an int n in [0, 8].  info["logprobs"] then holds the model's log-probability of every
        token in `tokens`, log_softmax(logits)[token] of the row that predicted it - no temperature, top-p or top-k, in
        greedy and sampled decoding alike; with `penalties`, of the penalized row the token was chosen from, so under
        greedy decoding top_logprobs[0] is the emitted token - and, for n > 0, info["top_logprobs"] the n most likely
        tokens at each of those positions as (token_id, logprob) pairs (value descending, lowest id first among equals).
        They are scored on the device from the logits the decode step already computed (one samd_token_logprobs launch
        per step and per admission); the tokens are the same as without.

        `penalties` (None: none): one Penalties for every request or a sequence with one per request - repetition,
        presence and frequency penalties applied to every logits row before verification (and before temperature,
        top-p and top-k when sampled).  A row is penalized from its own context: the prompt, the tokens emitted so far
        and the draft tokens on its path, so greedy decoding stays lossless against plain penalized greedy decoding.
        Tree mode (tree=) is allowed; its successor table then learns from penalized rows, which changes drafts, not
        tokens.  Neutral Penalties() give the tokens of penalties=None.

        info["finish_reason"] says why a request ended: "stop" (EOS or a stop sequence), "length" (max_new_tokens) or
        "cache" (a step could run past max_cache_len).  `stop` (None: none): one StopSequences for every request or a
        sequence with one per request.  The output ends at the earliest output position where one of the request's
        sequences ends - the prompt is never matched, a sequence may end inside a step or straddle two - so `tokens`
        (and `logprobs`) are a prefix of what the request emits without stop, ending with the matched tokens;
        info["stop_index"] is the index of the matched sequence in the request's list (the lowest among those ending
        there), None when none ended it.  A sequence that would complete after max_new_tokens does not fire; one that
        ends on EOS does.  The match runs on the device in the step (one samd_stop_match launch), so a stopped request
        frees its slot and emits nothing more from that step on.

        `controls` (None: none): one LogitControls for every request or a sequence with one per request - a logit bias,
        bad words and min_tokens (min_tokens <= the request's max_new_tokens), applied to every logits row after the
        penalties and before temperature, top-p and top-k: first the bias, then the bans.  Each draft row is controlled
        from its own context (the output so far and the draft tokens on its path) and the output position it predicts
        (a row at path depth d predicts out_len + d + 1), so greedy decoding stays lossless against plain controlled
        greedy decoding; the first token comes from the prompt's last row controlled as position 0.  All modes are
        allowed; in tree mode the successor table learns from controlled rows (drafts change, tokens do not), and
        logprobs are those of the controlled rows.  Neutral LogitControls() give the tokens of controls=None.  One
        samd_apply_logit_controls launch per step and one per admission batch."""
        logprobs = _check_logprobs(logprobs)
        self.serve_stats = None
        if hasattr(max_new_tokens, "__len__"):
            limits = [int(x) for x in max_new_tokens]
            max_limit = max(limits, default=1)
        else:
            limits, max_limit = None, int(max_new_tokens)
        V = self.lm.config.vocab_size
        reqs = self._with_sampling(self._requests(prompts, max_new_tokens if limits is None else limits), sampling)
        reqs = self._with_controls(self._with_stops(self._with_penalties(reqs, penalties), stop, V), controls, V)
        for i, tokens, hist, slot, lp, reason, hit in self._run(reqs, max(max_limit, 1), graph, check_every,
                                                                sampling is not None, logprobs, penalties is not None,
                                                                stop is not None, controls is not None):
            info = {"slot": slot, "accept_lengths": hist, "finish_reason": reason}
            if stop is not None:
                info["stop_index"] = hit
            if self._prefixes is not None:
                info["prefix_len"] = self._slot_plen[slot]
            if lp is not None:
                info["logprobs"] = lp[0]
                if logprobs:
                    info["top_logprobs"] = lp[1]
            yield i, tokens, info
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

    def _with_sampling(self, requests: Iterator[tuple], sampling) -> Iterator[tuple]:
        """(index, prompt, limit, SamplingParams or None) of every request: its own params (seed + index for one shared
        SamplingParams), checked as it is pulled.  Tree mode is refused at once."""
        if sampling is not None and getattr(self, "tree", None) is not None:
            raise K.SamdError("sampling is not supported in Token-Recycle tree mode (tree=): its table update rides on "
                              "the greedy verify launch")
        shared = sampling is None or isinstance(sampling, SamplingParams)
        return self._sampled_requests(requests, sampling if shared else list(sampling), shared)

    @staticmethod
    def _sampled_requests(requests: Iterator[tuple], sampling, shared: bool) -> Iterator[tuple]:
        for i, p, limit in requests:
            if sampling is None:
                yield i, p, limit, None
                continue
            if shared:
                sp = dataclasses.replace(sampling, seed=sampling.seed + i) if isinstance(sampling.seed, int) else sampling
            elif i >= len(sampling):
                raise K.SamdError(f"request {i}: sampling has {len(sampling)} values, fewer than the prompts")
            else:
                sp = sampling[i]
            if not isinstance(sp, SamplingParams):
                raise K.SamdError(f"request {i}: sampling must be a SamplingParams, got {type(sp).__name__}")
            bad = sp.problem()
            if bad:
                raise K.SamdError(f"request {i}: {bad}")
            yield i, p, limit, sp

    @staticmethod
    def _with_penalties(requests: Iterator[tuple], penalties) -> Iterator[tuple]:
        """(index, prompt, limit, SamplingParams or None, Penalties or None) of every request: the shared Penalties or
        its own, checked as it is pulled."""
        shared = penalties is None or isinstance(penalties, Penalties)
        if not shared:
            try:
                penalties = list(penalties)
            except TypeError:
                raise K.SamdError(f"penalties must be None, a Penalties or a sequence of them, got "
                                  f"{type(penalties).__name__}") from None
        for i, p, limit, sp in requests:
            if penalties is None:
                yield i, p, limit, sp, None
                continue
            if shared:
                pn = penalties
            elif i >= len(penalties):
                raise K.SamdError(f"request {i}: penalties has {len(penalties)} values, fewer than the prompts")
            else:
                pn = penalties[i]
            if not isinstance(pn, Penalties):
                raise K.SamdError(f"request {i}: penalties must be a Penalties, got {type(pn).__name__}")
            bad = pn.problem()
            if bad:
                raise K.SamdError(f"request {i}: {bad}")
            yield i, p, limit, sp, pn

    @staticmethod
    def _with_stops(requests: Iterator[tuple], stop, vocab: int) -> Iterator[tuple]:
        """(index, prompt, limit, SamplingParams or None, Penalties or None, StopSequences or None) of every request: the
        shared StopSequences or its own, checked against the vocabulary as it is pulled."""
        shared = stop is None or isinstance(stop, StopSequences)
        if not shared:
            try:
                stop = list(stop)
            except TypeError:
                raise K.SamdError(f"stop must be None, a StopSequences or a sequence of them, got "
                                  f"{type(stop).__name__}") from None
        for i, p, limit, sp, pn in requests:
            if stop is None:
                yield i, p, limit, sp, pn, None
                continue
            if shared:
                ss = stop
            elif i >= len(stop):
                raise K.SamdError(f"request {i}: stop has {len(stop)} values, fewer than the prompts")
            else:
                ss = stop[i]
            if not isinstance(ss, StopSequences):
                raise K.SamdError(f"request {i}: stop must be a StopSequences, got {type(ss).__name__}")
            bad = ss.problem(vocab)
            if bad:
                raise K.SamdError(f"request {i}: {bad}")
            yield i, p, limit, sp, pn, ss

    @staticmethod
    def _with_controls(requests: Iterator[tuple], controls, vocab: int) -> Iterator[tuple]:
        """(index, prompt, limit, SamplingParams or None, Penalties or None, StopSequences or None, LogitControls or None)
        of every request: the shared LogitControls or its own, checked against the vocabulary and the request's
        max_new_tokens as it is pulled."""
        shared = controls is None or isinstance(controls, LogitControls)
        if not shared:
            try:
                controls = list(controls)
            except TypeError:
                raise K.SamdError(f"controls must be None, a LogitControls or a sequence of them, got "
                                  f"{type(controls).__name__}") from None
        for i, p, limit, sp, pn, ss in requests:
            if controls is None:
                yield i, p, limit, sp, pn, ss, None
                continue
            if shared:
                lc = controls
            elif i >= len(controls):
                raise K.SamdError(f"request {i}: controls has {len(controls)} values, fewer than the prompts")
            else:
                lc = controls[i]
            if not isinstance(lc, LogitControls):
                raise K.SamdError(f"request {i}: controls must be a LogitControls, got {type(lc).__name__}")
            bad = lc.problem(vocab)
            if bad:
                raise K.SamdError(f"request {i}: {bad}")
            if lc.min_tokens > limit:
                raise K.SamdError(f"request {i}: min_tokens {lc.min_tokens} exceeds max_new_tokens {limit}")
            yield i, p, limit, sp, pn, ss, lc


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
    read per `check_every` steps, generate() and serve()) is BatchedSamdDecoder's, and so is prefix reuse
    (max_prefixes, add_prefix, drop_prefix): a registered prefix carries its automaton and static cursor, so the static
    trees of a request that starts from one are those of its full prompt.  stats["tree_steps"] (and
    serve_stats["tree_steps"]) counts the request-steps of live requests that drafted a static tree.

    Known corner, inherited from the reference (SURVEY Appendix A9): a -1 pad column of a path selects token 0, so it is
    "accepted" when the compared row's argmax is token 0, and the KV move then copies row cache_len - 1.  The batched path
    table is D wide while a reference tree is only as wide as its own deepest path (and a reference sequence as long as
    its draft), so here pads beyond a request's own width can be compared too - only after every real node of the path
    was accepted, i.e. when the LM's greedy next token is 0.  A sampled call (sampling=...) verifies every request only up
    to its own width (samd_verify_sample_requests with the longest path of its row of the table), then samd_kv_compact
    moves its accepted rows: there the pads beyond a request's own draft are never compared."""

    def __init__(self, lm, batch: int, max_cache_len: int, max_predicts: int = 40, alpha: float = 4.0, K: int = 8,
                 len_bias: int = 5, static: Optional[E.StaticSamDevice] = None, eos_token_id: Optional[int] = None,
                 max_tokens: int = 16384, dtype=torch.float16, device="cuda", max_prefixes: int = 0):
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
                        n_nodes=mk(batch), n_paths=mk(batch), retrieve=mk(batch, T, T), depth=mk(batch),
                        mask=torch.zeros(batch * T * max_cache_len, dtype=dtype, device=dev))
        self._init_pool(max_prefixes)

    def _extra_state(self, mk) -> dict:
        return dict(tree_steps=torch.zeros(1, dtype=torch.long, device=self.device))

    def _extra_stats(self) -> dict:
        return dict(tree_steps=int(self._st["tree_steps"].item()))

    def mask_view(self, kv_len: int) -> torch.Tensor:
        return self.buf["mask"][:self.B * self.T * kv_len].view(self.B, self.T, kv_len)

    def _draft_forward_verify(self, kv_len: int) -> tuple:
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
                         attention_mask=mask[:, None]).logits.contiguous()
        self._penalize(logits, buf["tokens"], buf["retrieve"], buf["n_nodes"], buf["n_paths"])
        self._control(logits, buf["tokens"], buf["retrieve"], buf["n_nodes"], buf["n_paths"])
        if self._sampled:
            # a request's own width - its draft length, or its tree's deepest path - so that the -1 pads beyond it are
            # never compared; then the accepted rows move into place
            torch.amax((buf["retrieve"] >= 0).sum(2, dtype=torch.int32), 1, out=buf["depth"])
            res = self._verify_sample(logits, buf["tokens"], buf["retrieve"], n_paths=buf["n_paths"],
                                      n_nodes=buf["n_nodes"], depth=buf["depth"])
            self.ver.kv_compact(res["indices"], res["accept_len"], cache.cache_len)
            return res, logits, buf["n_nodes"]
        return self.ver.verify(logits, buf["tokens"], buf["retrieve"], cache_len=cache.cache_len, move_kv=True,
                               n_nodes=buf["n_nodes"], n_paths=buf["n_paths"], out=st["res"]), logits, buf["n_nodes"]
