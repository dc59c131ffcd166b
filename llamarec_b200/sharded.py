"""Row-sharded multi-GPU retrieval (north_star: item table sharded by row range across the GPUs of one
box, local top-k per rank, one all-gather over NVLink, k-way merge kernel).

The reference has no multi-device retrieval path (SURVEY section 2.1); its single-device result is the
oracle: merging exact per-shard top-k lists reproduces the unsharded top-k exactly.

One process per GPU (`torch.distributed`, NCCL).  Per batch:
  1. every rank encodes its slice of the users (the encoder is batch-sharded: replicated encode would
     be the Amdahl term at 8 GPUs) and all-gathers the 64-d user states            [B x 64 fp32]
  2. every rank scores ALL users against ITS item rows and keeps a local top-k     (no communication)
  3. ONE all-gather of the local lists, scores and ids packed in one payload       [R x 2 x B x k x 4 bytes]
  4. every rank merges the R lists (fused with the metrics)                        (no communication)

Two batch layouts are supported:
  * `retrieve(x)`     -- every rank passes the SAME batch (strong scaling: fixed batch, fixed catalogue);
  * `retrieve_dp(x)`  -- every rank passes ITS OWN batch of b users (data-parallel users x row-sharded items,
                         weak scaling: the global batch is R*b).  Per step:
      1. encode the local users; ONE coalesced all-gather of (user state, exclusion list, filter)
      2. score all R*b users against the local item rows, local top-k              (no communication)
      3. ONE all-to-all: the lists of rank j's users go to rank j                   [R x b x 2 x k x 4 bytes]
      4. merge the R lists of the local users (fused with the metrics)             (no communication)

On NVLink (NCCL process group + CUDA backend) steps 1 and 3 of `retrieve_dp` do not go through a collective
library at all: every rank STORES its exchange records into its slot of every peer's gather buffer
(`lrb_peer_push`), and the local merge kernel scatters each user's list straight into the recv buffer of
the rank that owns the user (`lrb_merge_metrics_scatter`) -- the transfer is the kernel's own epilogue.
The buffers live in symmetric memory (peer-mapped over NVLink/NVSwitch), are double buffered, and one
signal-pad barrier per exchange orders the ranks.  Without symmetric memory (gloo on CPU in the tests) the
same step runs on `all_gather_into_tensor` / `all_to_all_single`.

The numerical work is delegated to a backend object so that the plumbing (ranges, padding, gather
layout) can be exercised on CPU with gloo in tests; the product backend drives the CUDA kernels.
"""
from __future__ import annotations

from typing import Dict, Optional, Sequence, Tuple

import torch
import torch.distributed as dist


def _check_k(k: int) -> None:
    # the exchange buffers and the scatter merge are built for the streaming kernels' lists
    if int(k) > 50:
        raise ValueError(f"row-sharded retrieval takes k <= 50, got k={k} (LRURec.retrieve takes up to 1024)")


def shard_range(n: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous split of range(n) into `world` pieces of ceil(n/world) (the last may be short/empty)."""
    per = (n + world - 1) // world
    lo = min(rank * per, n)
    return lo, min(lo + per, n)


class CudaBackend:
    """Product backend: llamarec_b200.LRURec restricted to this rank's row shard."""

    def __init__(self, model, rank: int, world: int, precision: str = "auto"):
        if precision == "exact":
            # _precision would resolve it to a per-shard choice; exact retrieval across row shards is not built
            raise ValueError('precision="exact" is not supported by the sharded backend (use LRURec.retrieve)')
        self.model = model
        # 'auto' is resolved ONCE from the whole catalogue, not from this rank's shard: shard_range gives the
        # last rank a shorter shard, and ranks that disagree would exchange states of different widths and
        # merge scores of different precisions
        prec = model._precision(precision, model.num_items + 1)
        self.precision = "fp32" if prec == 1 else "bf16"
        self._packed = {}
        lo, hi = shard_range(model.num_items + 1, rank, world)
        model.set_row_shard(lo, hi)
        self.rows = (lo, hi)

    def encode(self, x: torch.Tensor) -> torch.Tensor:
        return self.model.encode(x)

    def local_topk_packed(self, x: torch.Tensor, u: torch.Tensor, k: int, exclude_history: bool) -> torch.Tensor:
        """Local top-k as ONE gather payload: int32 [2, B, k] = scores (bit pattern), ids."""
        _check_k(k)
        B = x.shape[0]
        key = (B, k, str(u.device))
        buf = self._packed.get(key)
        if buf is None:
            buf = torch.empty(2, B, k, dtype=torch.int32, device=u.device)
            self._packed[key] = buf
        if self.rows[1] <= self.rows[0]:   # empty shard (more ranks than rows): nothing to offer
            buf[0].view(torch.float32).fill_(float("-inf"))
            buf[1].fill_(-1)
            return buf
        self.model.retrieve(x, k=k, exclude_history=exclude_history, precision=self.precision, u=u, packed_out=buf,
                            packed_layout="planes")
        return buf

    # ---- data-parallel users (retrieve_dp) ----
    def encode_states(self, x: torch.Tensor, exclude_history: bool):
        """Local users -> what the other ranks need to score them: user state [b, 64] (bf16 for the tensor-core
        path, fp32 for the exact path), sorted exclusion list [b, stride] and its filter [b, 4]."""
        m = self.model
        rows = m.row_end - m.row_begin
        prec = m._precision(self.precision, max(rows, 1))
        x = x.to(m.embedding.token.weight.device).contiguous()
        seq = m._prepare_sequences(x, all_positions=False, want_excl=exclude_history)
        u, u16, _ = m._encode(x, all_positions=False, want_bf16=(prec == 0), seq=seq)
        return {"state": u16 if prec == 0 else u, "excl": seq["excl_sorted"], "bloom": seq["excl_bloom"],
                "excl_stride": seq["excl_stride"], "u": u}

    supports_peer_exchange = True

    def local_topk_rows(self, state: torch.Tensor, excl, bloom, excl_stride: int, k: int,
                        scatter: Optional[dict] = None) -> Optional[torch.Tensor]:
        """All R*b users against this rank's rows -> int32 [R*b, 2, k]: per user scores (bit pattern), ids.
        With `scatter` the rows are written into the owners' recv buffers instead (nothing is returned)."""
        _check_k(k)
        B = state.shape[0]
        if scatter is not None and self.rows[1] > self.rows[0]:
            seq = {"excl_sorted": excl, "excl_bloom": bloom, "excl_stride": excl_stride}
            kw = {"u_bf16": state} if state.dtype == torch.bfloat16 else {"u": state}
            self.model.retrieve(None, k=k, exclude_history=excl is not None, precision=self.precision, seq=seq,
                                scatter=scatter, **kw)
            return None
        key = ("rows", B, k, str(state.device))
        buf = self._packed.get(key)
        if buf is None:
            buf = torch.empty(B, 2, k, dtype=torch.int32, device=state.device)
            self._packed[key] = buf
        if self.rows[1] <= self.rows[0]:
            buf.view(torch.float32)[:, 0].fill_(float("-inf"))
            buf[:, 1].fill_(-1)
            return buf
        seq = {"excl_sorted": excl, "excl_bloom": bloom, "excl_stride": excl_stride}
        kw = {"u_bf16": state} if state.dtype == torch.bfloat16 else {"u": state}
        self.model.retrieve(None, k=k, exclude_history=excl is not None, precision=self.precision, seq=seq,
                            packed_out=buf, packed_layout="per_user", **kw)
        return buf

    def merge_rows(self, recv: torch.Tensor, k, labels, ks):
        """recv: int32 [R, b, 2, k] (row j = rank j's lists for the local users) -> final lists (+ metrics)."""
        from .model import merge_lists
        R, b, _, K = recv.shape
        scores = recv.view(torch.float32)[:, :, 0]
        ids = recv[:, :, 1]
        return merge_lists(scores, ids, None, k_out=k, labels=labels, ks=ks, layout="list_major",
                           strides=(b * 2 * K, 2 * K))

    def merge_packed(self, gathered: torch.Tensor, k, labels, ks):
        """gathered: int32 [R, 2, B, k] (all-gathered payloads) -> final lists (+ metrics)."""
        from .model import merge_lists
        R, _, B, K = gathered.shape
        scores = gathered[:, 0].view(torch.float32)
        ids = gathered[:, 1]
        # missing entries carry id -1 / score -inf and simply never win
        return merge_lists(scores, ids, None, k_out=k, labels=labels, ks=ks, layout="list_major",
                           strides=(2 * B * K, K))


class PeerExchange:
    """Symmetric-memory buffers of one (b, k, record layout) configuration: per parity a gather region
    (state | exclusion list | filter, R*b rows each) and a recv region [R][b][2][k] int32."""

    def __init__(self, group, rank: int, world: int, device, b: int, k: int, rec_bytes: Sequence[int]):
        import torch.distributed._symmetric_memory as symm
        self.rank, self.world, self.b, self.k = rank, world, b, k
        self.rec_bytes = list(rec_bytes)
        al = lambda n: (n + 255) // 256 * 256
        off = 0
        self.gather_off, self.recv_off = [], []
        for _ in range(2):
            offs = []
            for rb in self.rec_bytes:
                offs.append(off)
                off += al(world * b * rb)
            self.gather_off.append(offs)
        for _ in range(2):
            self.recv_off.append(off)
            off += al(world * b * 2 * k * 4)
        self.total = off
        self.parity = 0     # which copy of the buffers the next step uses (all ranks step together)
        self.buf = symm.empty(self.total, dtype=torch.uint8, device=device)
        name = (group if group is not None else dist.group.WORLD).group_name
        self.hdl = symm.rendezvous(self.buf, name)
        self.ptrs = [int(p) for p in self.hdl.buffer_ptrs]

    def barrier(self, channel: int) -> None:
        self.hdl.barrier(channel=channel)

    def gather_view(self, parity: int, a: int, dtype, row_shape) -> torch.Tensor:
        n = self.world * self.b * self.rec_bytes[a]
        o = self.gather_off[parity][a]
        return self.buf[o:o + n].view(dtype).view((self.world * self.b,) + tuple(row_shape))

    def recv_view(self, parity: int) -> torch.Tensor:
        n = self.world * self.b * 2 * self.k * 4
        o = self.recv_off[parity]
        return self.buf[o:o + n].view(torch.int32).view(self.world, self.b, 2, self.k)


class ShardedRetriever:
    def __init__(self, backend, group: Optional[dist.ProcessGroup] = None, exchange: str = "auto"):
        """exchange: 'peer' (stores into symmetric memory, needs NCCL + CUDA), 'collective'
        (torch.distributed all-gather / all-to-all), or 'auto' (peer when available)."""
        self.backend = backend
        self.group = group
        if exchange not in ("auto", "peer", "collective"):
            raise ValueError(f"unknown exchange {exchange!r}")
        self.exchange = exchange
        self._peer = {}
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self._bufs = {}
        self.phase_events = None     # optional list: retrieve_dp appends (phase name, CUDA event) pairs
        self._coalesce = dist.is_initialized() and dist.get_backend(group) == "nccl"

    def _all_gather(self, t: torch.Tensor) -> torch.Tensor:
        if self.world == 1:
            return t.unsqueeze(0)
        t = t.contiguous()
        out = torch.empty((self.world * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
        dist.all_gather_into_tensor(out, t, group=self.group)   # concatenated along dim 0 (gloo and nccl)
        return out.reshape((self.world,) + tuple(t.shape))

    def _mark(self, name: str) -> None:
        if self.phase_events is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            self.phase_events.append((name, ev))

    def _peer_exchange(self, b: int, k: int, st: dict) -> Optional[PeerExchange]:
        if self.exchange == "collective" or not getattr(self.backend, "supports_peer_exchange", False):
            return None
        if self.exchange == "auto" and not (dist.is_initialized() and dist.get_backend(self.group) == "nccl"):
            return None
        if self.exchange == "auto" and self.world > 16:      # lrb_peer_push / scatter address <= 16 destinations
            return None
        arrays = [t for t in (st["state"], st["excl"], st["bloom"]) if t is not None]
        rec = tuple(t[0].numel() * t.element_size() for t in arrays)
        key = (b, k, rec, str(arrays[0].dtype))
        if key not in self._peer:
            try:
                self._peer[key] = PeerExchange(self.group, self.rank, self.world, arrays[0].device, b, k, rec)
            except Exception as e:                      # symmetric memory not available on this system
                if self.exchange == "peer":
                    raise
                import warnings
                warnings.warn(f"peer-memory exchange unavailable ({e!r}); using torch.distributed collectives")
                self._peer[key] = None
        return self._peer[key]

    def _retrieve_dp_peer(self, px: PeerExchange, st: dict, b: int, k: int, labels, ks):
        from . import _lib
        lib = _lib.load()
        mark = self._mark
        par = px.parity
        px.parity ^= 1
        arrays = [t for t in (st["state"], st["excl"], st["bloom"]) if t is not None]
        n_arr, R = len(arrays), self.world
        # 1. all-gather by stores: my b records go to slot `rank` of every rank's gather region
        src = (_lib.ctypes.c_void_p * n_arr)(*[t.data_ptr() for t in arrays])
        nbytes = (_lib.ctypes.c_size_t * n_arr)(*[b * rb for rb in px.rec_bytes])
        dst = (_lib.ctypes.c_void_p * (n_arr * R))(*[
            px.ptrs[d] + px.gather_off[par][a] + self.rank * b * px.rec_bytes[a]
            for a in range(n_arr) for d in range(R)])
        with _lib.on_device(arrays[0]):
            _lib.check(lib.lrb_peer_push(src, nbytes, n_arr, dst, R, _lib.stream_handle()))
        px.barrier(0)
        mark("all_gather")
        # 2. score all R*b users against the local rows; the local merge scatters each user's list to its owner
        views = [px.gather_view(par, a, t.dtype, t.shape[1:]) for a, t in enumerate(arrays)]
        state = views[0]
        excl, bloom = (views[1], views[2]) if st["excl"] is not None else (None, None)
        base = [px.ptrs[d] + px.recv_off[par] + self.rank * b * 2 * k * 4 for d in range(R)]
        scatter = {"dst_scores": base, "dst_ids": [p + k * 4 for p in base], "users_per_dst": b,
                   "out_stride": 2 * k}
        rows = self.backend.local_topk_rows(state, excl, bloom, st["excl_stride"], k, scatter=scatter)
        if rows is not None:                                # empty shard: nothing was scattered, hand out the fill
            for d in range(R):
                px.hdl.get_buffer(d, (px.total,), torch.uint8)[
                    px.recv_off[par] + self.rank * b * 2 * k * 4:][:b * 2 * k * 4].view(torch.int32).copy_(
                    rows[d * b:(d + 1) * b].reshape(-1))
        mark("score+local_merge")
        px.barrier(1)
        mark("all_to_all")
        # 3. merge the R lists of the local users
        out = self.backend.merge_rows(px.recv_view(par), k, labels, ks)
        mark("merge")
        out["u"] = st["u"]
        return out

    def _all_gather_many(self, tensors):
        """All-gathers several per-rank tensors (None entries pass through) as ONE collective launch where the
        backend can coalesce them (NCCL group), else one after the other.  Outputs are [R*b, ...]."""
        if self.world == 1:
            return list(tensors)
        outs = []
        for i, t in enumerate(tensors):
            if t is None:
                outs.append(None)
                continue
            key = ("ag", i, tuple(t.shape), t.dtype, str(t.device))
            o = self._bufs.get(key)
            if o is None:
                o = torch.empty((self.world * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
                self._bufs[key] = o
            outs.append(o)
        pairs = [(o, t.contiguous()) for o, t in zip(outs, tensors) if t is not None]
        if self._coalesce and len(pairs) > 1:
            try:
                with dist._coalescing_manager(group=self.group, device=pairs[0][1].device, async_ops=False):
                    for o, t in pairs:
                        dist.all_gather_into_tensor(o, t, group=self.group)
                return outs
            except (RuntimeError, NotImplementedError, AttributeError, TypeError):
                self._coalesce = False       # backend without coalescing support: plain calls from now on
        for o, t in pairs:
            dist.all_gather_into_tensor(o, t, group=self.group)
        return outs

    @torch.no_grad()
    def retrieve_dp(self, x: torch.Tensor, k: int = 20, exclude_history: bool = True,
                    labels: Optional[torch.Tensor] = None, ks: Optional[Sequence[int]] = None) -> Dict[str, torch.Tensor]:
        """x: THIS rank's users [b, L] (every rank passes the same b; labels likewise [b]).  Returns the final
        top-k of the local users against the WHOLE catalogue (+ metric sums over the local users)."""
        _check_k(k)
        b = x.shape[0]
        mark = self._mark
        mark("begin")
        st = self.backend.encode_states(x, exclude_history)
        mark("encode")
        px = self._peer_exchange(b, k, st) if self.world > 1 else None
        if px is not None:
            return self._retrieve_dp_peer(px, st, b, k, labels, ks)
        state, excl, bloom = self._all_gather_many([st["state"], st["excl"], st["bloom"]])
        mark("all_gather")
        payload = self.backend.local_topk_rows(state, excl, bloom, st["excl_stride"], k)      # [R*b, 2, k]
        mark("score+local_merge")
        if self.world > 1:
            key = ("a2a", tuple(payload.shape), str(payload.device))
            recv = self._bufs.get(key)
            if recv is None:
                recv = torch.empty_like(payload)
                self._bufs[key] = recv
            dist.all_to_all_single(recv, payload, group=self.group)
        else:
            recv = payload
        mark("all_to_all")
        out = self.backend.merge_rows(recv.view(self.world, b, 2, k), k, labels, ks)
        mark("merge")
        out["u"] = st["u"]
        return out

    @torch.no_grad()
    def retrieve(self, x: torch.Tensor, k: int = 20, exclude_history: bool = True,
                 labels: Optional[torch.Tensor] = None, ks: Optional[Sequence[int]] = None) -> Dict[str, torch.Tensor]:
        """x: the FULL batch of id sequences [B, L], identical on every rank."""
        _check_k(k)
        B = x.shape[0]
        per = (B + self.world - 1) // self.world
        lo, hi = shard_range(B, self.rank, self.world)
        # 1. batch-sharded encode, padded to a common slice size for the collective
        u_loc = torch.zeros(per, 64, dtype=torch.float32, device=x.device)
        if hi > lo:
            u_loc[: hi - lo] = self.backend.encode(x[lo:hi])
        u = self._all_gather(u_loc).reshape(self.world * per, 64)[:B].contiguous()
        # 2. local scoring over this rank's rows -> one packed payload [2, B, k] (scores, ids)
        payload = self.backend.local_topk_packed(x, u, k, exclude_history)
        # 3. ONE all-gather of the (score, id) lists
        gathered = self._all_gather(payload)
        # 4. merge (+ metrics)
        out = self.backend.merge_packed(gathered, k, labels, ks)
        out["u"] = u
        return out
