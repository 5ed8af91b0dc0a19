"""Dictionary-sharded b_sae for 2^20-latent dictionaries (BASELINE config 5, SURVEY.md 8e).

The reference BinarySAE (sae/binary.py:73-103) keeps the whole dictionary in one process. Here rank
g of G owns the latents [g*H/G, (g+1)*H/G): its slice of encoder.0.weight / bias and of the bit-plane
logits decoder.weight; decoder.bias and the input batch x are replicated. One forward is

    local fused encoder + top-k over the shard  (tcgen05 kernel, shard-local indices)
    all-gather of the (value, index) candidates  -> [G, B, k] on every rank            (collective 1)
        (large k: k / G + 6 sigma candidates per shard first; the merge verifies that no shard ran out of
         candidates and the exchange is repeated with the full k only then -- ShardPlan.k_send)
    merge to the global top-k, (value desc, global index asc): identical on every rank
    sparse decode of the winners this shard owns -> partial reconstruction [B, D]
    reduce-scatter(sum) of the partials          -> this rank's B/G rows of the result (collective 2)

which equals the reference forward on the concatenated dictionary: topk over all H latents
(:94) and latent.matmul(int_weights) (:38) split by rows of int_weights.

DictionaryShardedBaselineSAE runs the same choreography for the top-k baseline (sae/baseline.py): its encoder is the
same fused encoder + top-k on raw pre-activations, and a shard decodes its winners from its columns of the
nn.Linear(H, D) decoder. Everything between the local top-k and the decode (the exchange rounds, the large-k retry,
the peer-exchange lifecycle, gather_output) lives once, in _DictionaryShardedForward; the ops object owns the
model-specific steps.

The baseline also trains sharded (`autograd = True`, _ShardedBaselineFn). Its gradients split by latent: grad W_enc[h],
grad b_enc[h] and grad W_dec[:, h] read only the entries that selected h, which the shard owning h can compute from the
global winners every rank holds. The backward is

    all-gather of d loss / d rows               -> g [B, D] on every rank           (the forward's reduce-scatter, adjointed)
    all-gather of d loss / d values, summed in rank order -> [B, k], the same bits on every rank
    the latent-major backward over this shard's latent range (qsae_baseline_backward_range)

and every shard gradient is bit-equal to the matching slice of the single-GPU backward; grad b_dec (the column sums of
g) is the full gradient, the same bits on every rank.

The collectives go through torch.distributed (NCCL over NVLink on the B200 box; gloo in the CPU
tests). The compute steps are injected as `ops`: `CudaShardOps` (libqsae_b200.so, the product) is the
default; the CPU tests pass a numpy implementation to exercise the choreography under gloo. There is
no CPU fallback in the product: CudaShardOps raises on non-CUDA tensors.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import torch
import torch.nn as nn

from . import _lib
from .sae.base import PreparedCache, invalidate_prepared, param_key
from .sparse import SparseLatents


@dataclass(frozen=True)
class ShardPlan:
    """Pure host-side partition arithmetic (covered by the CPU tests)."""
    hidden_dim: int
    world_size: int
    rank: int

    def __post_init__(self):
        if self.world_size < 1 or not (0 <= self.rank < self.world_size):
            raise ValueError(f"bad rank {self.rank} / world size {self.world_size}")
        if self.hidden_dim % self.world_size != 0:
            raise ValueError(f"hidden_dim {self.hidden_dim} is not divisible by the world size {self.world_size}")

    @property
    def shard_latents(self) -> int:
        return self.hidden_dim // self.world_size

    @property
    def latent_begin(self) -> int:
        return self.rank * self.shard_latents

    def latent_range(self, rank: int | None = None) -> tuple:
        r = self.rank if rank is None else rank
        return r * self.shard_latents, (r + 1) * self.shard_latents

    def k_local(self, k: int) -> int:
        """Candidates each shard contributes: its own top-min(k, shard size) contains every global winner it owns."""
        return min(k, self.shard_latents)

    def k_send(self, k: int, min_k: int = 256) -> int:
        """Candidates a shard sends in the first exchange round. A shard owns ~k / G of a row's winners (latents are
        not ordered by importance), so for large k its top k / G + 6 sqrt(k / G) + 16 almost always covers its share:
        2097 -> 376 per shard at G = 8, which cuts the all-gather and the merge input 5.6x. The merge verifies it
        (a shard whose whole list was selected may hold more) and the exchange is repeated with k_local on failure."""
        kl = self.k_local(k)
        if self.world_size == 1 or k < min_k:
            return kl
        share = k / self.world_size
        return min(kl, int(math.ceil(share + 6.0 * math.sqrt(share) + 16)))

    def padded_batch(self, batch: int) -> int:
        """reduce-scatter needs equal row blocks: the batch is padded to a multiple of the world size."""
        return -(-batch // self.world_size) * self.world_size

    def row_range(self, batch: int, rank: int | None = None) -> tuple:
        """Rows of the (unpadded) batch whose reconstruction lands on `rank` after the reduce-scatter."""
        r = self.rank if rank is None else rank
        per = self.padded_batch(batch) // self.world_size
        return min(batch, r * per), min(batch, (r + 1) * per)

    def shard_state_dict(self, full: dict, n_bits: int) -> dict:
        """Slice a full BinarySAE state_dict (sae/binary.py layout) down to this rank's shard."""
        a, b = self.latent_range()
        return {"encoder.0.weight": full["encoder.0.weight"][a:b].clone(),
                "encoder.0.bias": full["encoder.0.bias"][a:b].clone(),
                "decoder.weight": full["decoder.weight"][a:b].clone(),
                "decoder.bias": full["decoder.bias"].clone()}

    def merge_baseline_state_dicts(self, shard_sds) -> dict:
        """The inverse of shard_baseline_state_dict: the state_dicts of ranks 0 .. G-1, in rank order, -> one
        BaselineSparseAutoencoder state_dict (encoder rows and decoder columns concatenated, rank 0's decoder.bias).
        Raises ValueError if the shards do not fit this plan or the replicated decoder.bias differs between them."""
        if len(shard_sds) != self.world_size:
            raise ValueError(f"expected {self.world_size} shard state_dicts, got {len(shard_sds)}")
        hs = self.shard_latents
        for r, sd in enumerate(shard_sds):
            if sd["encoder.0.weight"].shape[0] != hs or sd["encoder.0.bias"].shape[0] != hs or sd["decoder.weight"].shape[1] != hs:
                raise ValueError(f"shard {r} does not hold {hs} latents")
        bias = shard_sds[0]["decoder.bias"]
        for r, sd in enumerate(shard_sds[1:], 1):
            if not torch.equal(sd["decoder.bias"], bias):
                raise ValueError(f"decoder.bias of rank {r} differs from rank 0's: the replicas diverged")
        return {"encoder.0.weight": torch.cat([sd["encoder.0.weight"] for sd in shard_sds], 0),
                "encoder.0.bias": torch.cat([sd["encoder.0.bias"] for sd in shard_sds], 0),
                "decoder.weight": torch.cat([sd["decoder.weight"] for sd in shard_sds], 1),
                "decoder.bias": bias.clone()}

    def shard_baseline_state_dict(self, full: dict) -> dict:
        """Slice a full BaselineSparseAutoencoder state_dict (sae/baseline.py layout) down to this rank's shard. The
        decoder is nn.Linear(H, D): its weight [D, H] is sliced by columns."""
        a, b = self.latent_range()
        return {"encoder.0.weight": full["encoder.0.weight"][a:b].clone(),
                "encoder.0.bias": full["encoder.0.bias"][a:b].clone(),
                "decoder.weight": full["decoder.weight"][:, a:b].clone(memory_format=torch.contiguous_format),
                "decoder.bias": full["decoder.bias"].clone()}


class _CudaEncoderOps:
    """The shard-local encoder + top-k and the candidate merge on libqsae_b200.so: the steps every dictionary-sharded
    module shares (the encoder is nn.Linear(D, H/G) on raw pre-activations in both)."""

    def __init__(self, module):
        self.m = module
        self._prep = PreparedCache()

    def _require_cuda(self, t: torch.Tensor) -> None:
        if not t.is_cuda:
            raise RuntimeError(f"{type(self.m).__name__} runs only on CUDA (no CPU fallback)")

    def _w_bf16(self):
        w = self.m.encoder[0].weight
        return self._prep.get("w_bf16", param_key(w), lambda: _lib.cast_bf16(w.detach().contiguous()))

    def _sample(self):
        lin = self.m.encoder[0]
        return self._prep.get("sample", param_key(lin.weight, lin.bias),
                              lambda: _lib.prepare_sample(self._w_bf16(), lin.bias.detach()))

    def local_topk(self, x: torch.Tensor, k_local: int):
        """-> (vals [B, k_local] f32, shard-local idx [B, k_local] i32)"""
        self._require_cuda(x)
        lin = self.m.encoder[0]
        w32 = lin.weight.detach().contiguous()
        vals, idx, _ = _lib.encode_topk(x, self._w_bf16(), w32 if self.m.exact else None, lin.bias.detach(), k_local,
                                        _lib.ACT_NONE, self.m.exact, sample=self._sample())
        return vals, idx

    def local_candidates(self, x: torch.Tensor, k_local: int) -> torch.Tensor:
        """-> [B, k_local, 2] int32 entries {value bits, shard-local index}"""
        return _lib.pack_candidates(*self.local_topk(x, k_local))

    def merge(self, cand_all: torch.Tensor, shard_latents: int, k: int, truncated: bool = False):
        return _lib.merge_candidates(cand_all, shard_latents, k, truncated=truncated)


class CudaShardOps(_CudaEncoderOps):
    """The compute steps of the dictionary-sharded b_sae on libqsae_b200.so."""

    def _packed(self):
        w = self.m.decoder_weight
        self._require_cuda(w)
        return self._prep.get("packed", param_key(w),
                              lambda: _lib.pack_bitplanes(w.detach(), self.m.input_dim, self.m.n_bits))

    def decode_partial(self, vals, idx, plan: ShardPlan, with_bias: bool, out: torch.Tensor | None = None) -> torch.Tensor:
        packed, _, gap = self._packed()
        if gap > self.m.polar_tol:
            raise RuntimeError("dictionary-sharded b_sae serves the packed (polarised / hard) dictionary only; "
                               f"max |sigmoid(w) - bit| = {gap:.3g} on this shard")
        return _lib.decode_range(vals, idx, packed, plan.shard_latents, plan.latent_begin, self.m.input_dim,
                                 self.m.quantization_step, self.m.decoder_bias.detach() if with_bias else None,
                                 self.m.n_bits, out=out)

    def polarize_numerator(self) -> float:
        """sum over the shard of p (1 - p) 2^i (sae/binary.py:41-42 before the mean)."""
        w = self.m.decoder_weight
        return self._packed()[1] * w.numel()


class CudaBaselineShardOps(_CudaEncoderOps):
    """The compute steps of the dictionary-sharded baseline_sae on libqsae_b200.so: the shared encoder and merge, and
    the decode of this shard's winners from its transposed fp32 decoder columns [H/G, D], cached per weight version
    as BaselineSparseAutoencoder._dec_rows does."""

    def _dec_rows(self):
        w = self.m.decoder.weight                     # [D, H/G]: feature vectors are columns
        self._require_cuda(w)
        return self._prep.get("dec_rows", param_key(w), lambda: _lib.transpose(w.detach().contiguous()))

    def decode_partial(self, vals, idx, plan: ShardPlan, with_bias: bool, out: torch.Tensor | None = None) -> torch.Tensor:
        return _lib.decode_rows_f32_range(vals, idx, self._dec_rows(), plan.latent_begin, 1.0,
                                          self.m.decoder.bias.detach() if with_bias else None, out=out)

    def backward_local(self, x, vals, idx, g, g_vals, plan: ShardPlan):
        """This shard's gradients from the global winners (vals, idx) [B, k], the gathered g = d loss / d recon [B, D]
        and the summed g_vals = d loss / d vals [B, k] -> (grad W_enc [H/G, D], grad b_enc [H/G], grad W_dec [D, H/G],
        grad b_dec [D] over the whole batch)."""
        return _lib.baseline_backward_range(x, vals, idx, g, g_vals, self._dec_rows(), plan.latent_begin)


class PeerExchange:
    """The two exchanges of the sharded forward over CUDA IPC peer memory (NVLink / NVSwitch) instead of NCCL.

    Every rank owns one buffer, mapped by all peers:
        [flags: 2 phases x G uint32][candidate lists: 2 slots x B x k x 8 B][partial rows: 2 slots x B x D x 4 B]
    A rank writes its own lists / partial rows, raises its sequence flag in every consumer's buffer, and the
    consumers read the data inside the merge / reduce kernels (P2P loads). Two slots: a rank can be one exchange
    ahead of the slowest reader, never two (its next publish is ordered after a merge that needed every peer's
    previous publish). Handles travel once, through the process group's object all-gather.

    Failure mode (the NCCL transport has none of its own: its watchdog owns that): a flag wait is bounded
    (QSAE_PEER_TIMEOUT_MS, default 20 s) and raises a device flag on expiry instead of hanging the GPU. The flag is
    copied to pinned host memory after every forward (asynchronously) and examined at the start of the next one and
    wherever the forward synchronises anyway: `check()` raises RuntimeError and marks the exchange broken, and the
    module drops it (results of the forward that timed out are invalid and the sequence numbers of the ranks no longer
    agree, so the exchange is rebuilt -- collectively -- on the next forward)."""

    FLAG_BYTES = 1024

    def __init__(self, dist, group, rank: int, world: int, device, max_rows: int, max_k: int, D: int):
        self.rank, self.world, self.device, self.D = rank, world, device, D
        self.max_rows, self.max_k = max_rows, max_k
        self.cand_slot = -(-(max_rows * max_k * 8) // 1024) * 1024
        self.part_slot = -(-(max_rows * D * 4) // 1024) * 1024
        self.cand_off = self.FLAG_BYTES
        self.part_off = self.cand_off + 2 * self.cand_slot
        nbytes = self.part_off + 2 * self.part_slot
        self.ptr, self.buf, handle = _lib.peer_alloc(nbytes, device)
        handles = [None] * world
        dist.all_gather_object(handles, handle, group=group)
        self.peer_ptrs = [self.ptr if g == rank else _lib.peer_import(handles[g]) for g in range(world)]
        i64 = dict(dtype=torch.int64, device=device)
        self.cand_bases = [torch.tensor([p + self.cand_off + s * self.cand_slot for p in self.peer_ptrs], **i64) for s in (0, 1)]
        self.part_bases = [torch.tensor([p + self.part_off + s * self.part_slot for p in self.peer_ptrs], **i64) for s in (0, 1)]
        self.signal_targets = [torch.tensor([p + (ph * world + rank) * 4 for p in self.peer_ptrs], **i64) for ph in (0, 1)]
        self.timed_out = torch.zeros((1,), dtype=torch.int32, device=device)
        self._host_flag = torch.zeros((1,), dtype=torch.int32).pin_memory()
        self._flag_event = None
        self.broken = False
        self._dist, self._group = dist, group
        self.seq = [0, 0]          # exchanges done per phase (identical on every rank)
        dist.barrier(group=group)  # every peer has mapped every buffer before the first signal is sent

    def fits(self, rows: int, k: int, D: int) -> bool:
        return rows <= self.max_rows and k <= self.max_k and D == self.D

    def _exchange(self, phase: int) -> int:
        """signal `my data of this exchange is in place`, wait for everybody's; -> slot that holds it"""
        self.seq[phase] += 1
        _lib.peer_signal(self.signal_targets[phase], self.seq[phase])
        _lib.peer_wait(self.ptr + phase * self.world * 4, self.world, self.seq[phase], self.timed_out)
        return (self.seq[phase] - 1) % 2

    def publish_candidates(self, vals: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
        """-> device int64 [G]: where the [B, k] lists of every shard start"""
        B, k = vals.shape
        slot = self.seq[0] % 2
        a = self.cand_off + slot * self.cand_slot
        _lib.pack_candidates(vals, idx, out=self.buf[a:a + B * k * 8].view(torch.int32).view(B, k, 2))
        assert self._exchange(0) == slot
        return self.cand_bases[slot]

    def partial_view(self, B: int) -> torch.Tensor:
        slot = self.seq[1] % 2
        a = self.part_off + slot * self.part_slot
        return self.buf[a:a + B * self.D * 4].view(torch.float32).view(B, self.D)

    def reduce_rows(self, row_begin: int, rows: int) -> torch.Tensor:
        slot = self._exchange(1)
        return _lib.reduce_partials_peer(self.part_bases[slot], row_begin, rows, self.D)

    def _raise(self):
        self.broken = True
        raise RuntimeError("peer exchange: a flag wait timed out (a peer did not publish its data within "
                           "QSAE_PEER_TIMEOUT_MS); the results of that forward are invalid")

    def check(self) -> None:
        """Synchronous check (one tiny device -> host read)."""
        if int(self.timed_out.item()) != 0:
            self._raise()

    def note_forward_done(self) -> None:
        """Queue an asynchronous copy of the timeout flag behind the forward that was just enqueued."""
        self._host_flag.copy_(self.timed_out, non_blocking=True)
        self._flag_event = torch.cuda.Event()
        self._flag_event.record()

    def check_previous(self) -> None:
        """No host synchronisation: looks at the flag copy of the previous forward if it has landed."""
        if self._flag_event is not None and self._flag_event.query():
            self._flag_event = None
            if int(self._host_flag[0]) != 0:
                self._raise()

    def close(self, collective: bool = True) -> None:
        """Unmap the peers' buffers, wait until every peer has unmapped ours (freeing memory that a peer still has
        mapped is undefined behaviour), then free. collective=False skips the barrier (teardown after a failure,
        when the peers may be gone)."""
        for g, p in enumerate(self.peer_ptrs):
            if g != self.rank:
                _lib.peer_close(p)
        self.peer_ptrs = []
        if collective:
            self._dist.barrier(group=self._group)
        _lib.peer_free(self.ptr)


class _DictionaryShardedForward(nn.Module):
    """The forward choreography shared by the dictionary-sharded modules: local top-k, candidate exchange (truncated
    round + full retry for large k), global merge, owner decode through `ops.decode_partial`, reduce of the partial
    rows, over NCCL collectives or peer memory. Subclasses own the parameters, `top_k()` and `ops`."""

    def __init__(self, hidden_dim, rank, world_size, process_group):
        super().__init__()
        import torch.distributed as dist

        self._dist = dist
        self.group = process_group
        if world_size is None:
            world_size = dist.get_world_size(process_group) if dist.is_initialized() else 1
        if rank is None:
            rank = dist.get_rank(process_group) if dist.is_initialized() else 0
        self.plan = ShardPlan(hidden_dim, world_size, rank)
        self.hidden_dim = hidden_dim
        self.exact = True
        self.gather_output = False
        self.trim_min_k = 256                # k below this: every shard sends its full top-k (tiny anyway)
        self.last_exchange = None            # "truncated" / "full": which candidate exchange produced the last forward
        self.last_k_send = None              # candidates per shard and row of the last (successful) exchange round
        self.transport = "nccl"              # "nccl" (torch.distributed collectives) | "p2p" (CUDA IPC peer memory)
        # False: the returned SparseLatents hold the k winners of each row as a SET (no value order). The reference only
        # uses them as a set (mask / scatter, sae/binary.py:96-99); sorting 2097 winners per row is most of the large-k
        # selection's instructions. Fast mode (exact = False) only; exact mode always sorts.
        self.ordered_latents = True
        self._peer = None

    def invalidate(self) -> None:
        """Forget the prepared copies of this shard's weights (needed after in-place edits through `.data`)."""
        invalidate_prepared(self)

    # ---- collectives (world size 1 degenerates to local views) -------------------------------
    def _all_gather(self, t: torch.Tensor) -> torch.Tensor:
        G = self.plan.world_size
        if G == 1:
            return t.unsqueeze(0)
        out = torch.empty((G * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
        self._dist.all_gather_into_tensor(out, t.contiguous(), group=self.group)
        return out.view((G,) + tuple(t.shape))

    def _reduce_scatter_rows(self, partial: torch.Tensor) -> torch.Tensor:
        G = self.plan.world_size
        if G == 1:
            return partial
        B, D = partial.shape
        Bp = self.plan.padded_batch(B)
        if Bp != B:
            partial = torch.cat([partial, partial.new_zeros((Bp - B, D))], 0)
        out = torch.empty((Bp // G, D), dtype=partial.dtype, device=partial.device)
        self._dist.reduce_scatter_tensor(out, partial.contiguous(), op=self._dist.ReduceOp.SUM, group=self.group)
        a, b = self.plan.row_range(B)
        return out[: b - a]

    def _gather_rows(self, rows: torch.Tensor, B: int) -> torch.Tensor:
        per = self.plan.padded_batch(B) // self.plan.world_size
        if rows.shape[0] != per:
            rows = torch.cat([rows, rows.new_zeros((per - rows.shape[0], rows.shape[1]))], 0)
        return self._all_gather(rows).reshape(-1, rows.shape[1])[:B]

    # ---- forward ------------------------------------------------------------------------------
    def _sharded_forward(self, x: torch.Tensor):
        """-> (SparseLatents over all H latents, this rank's reconstruction rows or all of them with gather_output)"""
        if x.dim() != 2 or x.shape[1] != self.input_dim:
            raise RuntimeError(f"expected a [batch, {self.input_dim}] matrix, got shape {tuple(x.shape)}")
        x = x.contiguous().float()
        k = self.top_k()
        if k > self.hidden_dim:
            raise RuntimeError(f"selected index k out of range (k={k} > H={self.hidden_dim})")
        if not self.ordered_latents and not self.exact and isinstance(self.ops, _CudaEncoderOps):
            with _lib.unordered_topk():
                return self._forward_impl(x, k)
        return self._forward_impl(x, k)

    def _forward_impl(self, x: torch.Tensor, k: int):
        plan, ops = self.plan, self.ops
        B = x.shape[0]
        k_loc, k_snd = plan.k_local(k), plan.k_send(k, self.trim_min_k)
        px = None
        if self.transport == "p2p" and plan.world_size > 1:
            px = self._peer_exchange(B, k_loc)
            px.check_previous()                # a flag wait of the previous forward timed out: raise before going on

        def exchange_and_merge(kk, truncated=False):
            if px is not None:
                bases = px.publish_candidates(*ops.local_topk(x, kk))
                return _lib.merge_candidates_peer(bases, B, kk, plan.shard_latents, k, truncated=truncated)
            cand_all = self._all_gather(ops.local_candidates(x, kk))         # [G, B, kk, 2]
            return ops.merge(cand_all, plan.shard_latents, k, truncated=truncated)  # global top-k, same on all ranks

        self.last_exchange = "full"
        vals = None
        if k_snd < k_loc:
            # round 1: truncated lists; every rank merges the same candidates and therefore sees the same verdict
            vals, idx, incomplete = exchange_and_merge(k_snd, truncated=True)
            if int(incomplete.item()) != 0:
                vals = None                                                   # some shard ran out of candidates
            else:
                self.last_exchange = "truncated"
            if px is not None:
                px.check()                     # the forward has synchronised anyway: a stale merge must not be used
        self.last_k_send = k_snd if vals is not None else k_loc
        if vals is None:
            vals, idx = exchange_and_merge(k_loc)
        with_bias = plan.rank == 0
        if px is not None:
            ops.decode_partial(vals, idx, plan, with_bias, out=px.partial_view(B))
            a, b = plan.row_range(B)
            rows = px.reduce_rows(a, b - a)
        else:
            rows = self._reduce_scatter_rows(ops.decode_partial(vals, idx, plan, with_bias))
        if self.gather_output and plan.world_size > 1:
            rows = self._gather_rows(rows, B)
        if px is not None:
            px.note_forward_done()
        return SparseLatents(vals, idx, (B, self.hidden_dim)), rows

    def local_candidates(self, x: torch.Tensor) -> torch.Tensor:
        """The rank-local stage alone (fused encoder sweep + top-k over this shard, candidates of the first exchange
        round): what bench.py times to split a step into local compute and exchange + merge + decode."""
        k = self.top_k()
        return self.ops.local_candidates(x.contiguous().float(), self.plan.k_send(k, self.trim_min_k))

    # ---- the same forward with both exchanges over peer memory --------------------------------------------------
    def _peer_exchange(self, rows: int, k: int) -> PeerExchange:
        if self._peer is not None and self._peer.broken:
            self._peer.close(collective=False)
            self._peer = None
        if self._peer is None or not self._peer.fits(rows, k, self.input_dim):
            if self._peer is not None:
                torch.cuda.synchronize()
                self._dist.barrier(group=self.group)      # nobody is still reading the old buffers
                self._peer.close()
            self._peer = PeerExchange(self._dist, self.group, self.plan.rank, self.plan.world_size, self.decoder.bias.device,
                                      rows, k, self.input_dim)
        return self._peer


class DictionaryShardedBinarySAE(_DictionaryShardedForward):
    """Rank-local shard of BinarySAE(input_dim, hidden_dim, gamma, n_bits) (sae/binary.py:73).

    state_dict keys are the reference's, with the latent axis sliced: encoder.0.weight [H/G, D],
    encoder.0.bias [H/G], decoder.weight [H/G, D*n_bits], decoder.bias [D] (replicated).
    forward(x) -> (SparseLatents over all H latents, recon rows owned by this rank [B/G, D] or the
    gathered [B, D] when `gather_output`, polarize_loss)."""

    def __init__(self, input_dim, hidden_dim, gamma=4.0, n_bits=8, *, rank=None, world_size=None,
                 process_group=None, ops=None):
        super().__init__(hidden_dim, rank, world_size, process_group)
        self.input_dim, self.n_bits, self.gamma = input_dim, n_bits, gamma
        self.quantization_step = gamma / (2 ** (n_bits - 1))
        self.k = 0.002
        hs = self.plan.shard_latents
        self.encoder = nn.Sequential(nn.Linear(input_dim, hs))
        self.decoder = nn.Module()
        self.decoder.weight = nn.Parameter(torch.empty(hs, input_dim * n_bits))
        self.decoder.bias = nn.Parameter(torch.zeros(input_dim))
        nn.init.xavier_uniform_(self.encoder[0].weight, gain=1)
        nn.init.zeros_(self.encoder[0].bias)
        nn.init.kaiming_normal_(self.decoder.weight)
        self.polar_tol = 1e-6
        self._pol_cache = None
        # ops=False defers the choice (tests install their own backend after construction)
        self.ops = CudaShardOps(self) if ops is None else (ops or None)

    @property
    def decoder_weight(self):
        return self.decoder.weight

    @property
    def decoder_bias(self):
        return self.decoder.bias

    def top_k(self) -> int:
        return int(self.hidden_dim * self.k)          # over the FULL dictionary, as sae/binary.py:94

    def polarize_loss(self, like: torch.Tensor) -> torch.Tensor:
        """mean over the FULL dictionary of p (1 - p) 2^i (sae/binary.py:41-42): weight-only, so the
        all-reduce of the per-shard numerators runs once per weight version, not per forward."""
        key = param_key(self.decoder.weight) + (str(like.device),)
        if self._pol_cache is None or self._pol_cache[0] != key:
            num = torch.tensor([self.ops.polarize_numerator()], dtype=torch.float64, device=like.device)
            if self.plan.world_size > 1:
                self._dist.all_reduce(num, group=self.group)
            total = self.hidden_dim * self.input_dim * self.n_bits
            self._pol_cache = (key, (num[0] / total).to(torch.float32))
        return self._pol_cache[1]

    def forward(self, x: torch.Tensor):
        latents, rows = self._sharded_forward(x)
        return latents, rows, self.polarize_loss(x)


class _ShardedBaselineFn(torch.autograd.Function):
    """(x, W_enc, b_enc, W_dec, b_dec) of one rank -> (values [B, k], indices [B, k], this rank's recon rows): the
    sharded forward behind one autograd node. The backward runs the same collectives on every rank, in a fixed order
    (see the module docstring), so every rank must run it."""

    @staticmethod
    def forward(ctx, x, w_enc, b_enc, w_dec, b_dec, module):
        ctx.set_materialize_grads(False)
        x = x.contiguous().float()
        lat, rows = module._sharded_forward(x)
        ctx.module = module
        ctx.save_for_backward(x, lat.values, lat.indices)
        ctx.mark_non_differentiable(lat.indices)
        return lat.values, lat.indices, rows

    @staticmethod
    def backward(ctx, g_vals, _g_idx, g_rows):
        m = ctx.module
        plan = m.plan
        x, vals, idx = ctx.saved_tensors
        B, D = x.shape
        a, b = plan.row_range(B)
        g_rows = (torch.zeros((b - a, D), dtype=torch.float32, device=x.device) if g_rows is None
                  else g_rows.detach().contiguous().float())
        g = m._gather_rows(g_rows, B).contiguous()                            # collective 1: g [B, D]
        gv = torch.zeros_like(vals) if g_vals is None else g_vals.detach().contiguous().float()
        if plan.world_size > 1:
            parts = m._all_gather(gv)                                         # collective 2: [G, B, k]
            gv = parts[0].clone()
            for r in range(1, plan.world_size):                               # rank order: the same bits on every run
                gv += parts[r]
        gwe, gbe, gwd, gbd = m.ops.backward_local(x, vals, idx, g, gv, plan)
        return None, gwe, gbe, gwd, gbd, None


class DictionaryShardedBaselineSAE(_DictionaryShardedForward):
    """Rank-local shard of BaselineSparseAutoencoder(input_dim, hidden_dim) (sae/baseline.py): the top-k baseline at
    2^20 latents, split over G ranks by latents.

    state_dict keys are the baseline's, with the latent axis sliced: encoder.0.weight [H/G, D], encoder.0.bias [H/G],
    decoder.weight [D, H/G] (the decoder is nn.Linear(H, D), so a shard holds a column slice), decoder.bias [D]
    (replicated, added by rank 0 only). ShardPlan.shard_baseline_state_dict slices a full checkpoint.

    forward(x) -> (SparseLatents over all H latents with global indices, recon rows): this rank's [B/G, D] rows after
    the reduce-scatter, or the gathered [B, D] with `gather_output`. There is no dense [B, H] latent (the single-GPU
    module's `return_dense`): at H = 2^20 and B = 4096 it would take 17 GB. `SparseLatents.to_dense()` builds it on
    request.

    Training: with `autograd = True` (not part of the state_dict) and grad mode on, the forward is the same forward
    behind one autograd node (_ShardedBaselineFn), and `lat.values` is differentiable. The objective is the SUM of the
    ranks' losses: each rank takes its loss on its own rows (rows of x in plan.row_range(B)), e.g.
    0.5 * ((rows - x[a:b]) ** 2).sum() / (B * D), plus any term on lat.values. After loss.backward() the .grad of
    encoder.0.weight, encoder.0.bias and decoder.weight is bit-equal to the single-GPU module's gradient of that
    objective sliced to this shard, and decoder.bias.grad is the full gradient, the same bits on every rank (replicated
    biases stay identical under any optimizer). EVERY rank must call backward() on a loss that depends on its rows: the
    backward's two all-gathers are unconditional and issued in a fixed order, and a rank that skips them hangs the
    others. Refused in training: gather_output (every rank would take its loss over the whole batch, counted G times)
    and an x that requires grad (its gradient would need an all-reduce). ShardPlan.merge_baseline_state_dicts joins
    the ranks' state_dicts into the single-GPU checkpoint layout."""

    def __init__(self, input_dim, hidden_dim, *, rank=None, world_size=None, process_group=None, ops=None):
        super().__init__(hidden_dim, rank, world_size, process_group)
        self.input_dim = input_dim
        hs = self.plan.shard_latents
        # nn.Linear's own initialisation of the shard; load a full checkpoint through shard_baseline_state_dict
        self.encoder = nn.Sequential(nn.Linear(input_dim, hs))
        self.decoder = nn.Linear(hs, input_dim)
        self.topk = 32
        # True: forward builds one autograd node (_ShardedBaselineFn) whenever grad mode is on
        self.autograd = False
        # ops=False defers the choice (tests install their own backend after construction)
        self.ops = CudaBaselineShardOps(self) if ops is None else (ops or None)

    def top_k(self) -> int:
        return int(self.topk)                         # a count over the FULL dictionary, as sae/baseline.py:35

    def forward(self, x: torch.Tensor):
        if not (self.autograd and torch.is_grad_enabled()):
            return self._sharded_forward(x)
        if self.gather_output:
            raise RuntimeError("DictionaryShardedBaselineSAE: gather_output is not supported in training (every rank would "
                               "hold the whole batch, and a loss over it would be counted once per rank)")
        if x.requires_grad:
            raise RuntimeError("DictionaryShardedBaselineSAE: x.requires_grad is not supported in training (x is "
                               "replicated: its gradient would need an all-reduce across the ranks)")
        lin, dec = self.encoder[0], self.decoder
        vals, idx, rows = _ShardedBaselineFn.apply(x, lin.weight, lin.bias, dec.weight, dec.bias, self)
        return SparseLatents(vals, idx, (x.shape[0], self.hidden_dim)), rows

    def normalize_decoder_weights(self):
        """Unit-norm decoder columns (sae/baseline.py:42-50). A column is one latent, so every norm is local to the
        shard that holds it: the single-GPU formula on the shard, with no collective."""
        with torch.no_grad():
            w = self.decoder.weight.data
            self.decoder.weight.data = w / torch.clamp(torch.norm(w, dim=0, keepdim=True), min=1e-8)
