"""Multi-GPU plumbing.  Trees and games are independent (cnode.cpp:415 touches tree i only; every
game owns its RNG, hanabi_game.h:114), so the root / game batch is split into contiguous ranges,
one process per GPU with a model replica, and the ONLY communication of a search is one
all_gather of the final root statistics over NCCL (84 B per tree at A=20)."""
import torch
import torch.distributed as dist


def shard_range(total, rank, world_size):
    """Contiguous range [lo, hi) of trees/games owned by `rank` (sizes differ by at most one)."""
    base, rem = divmod(int(total), int(world_size))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def wave_rows(visits, values, world, wave, position):
    """One ticket's rows of a gathered search wave (mcts.SearchPipeline(wave=G)): every rank contributes G * n rows,
    ticket `position` owns rows [position * n, (position + 1) * n) of each.  visits [world * G * n, A] and values
    [world * G * n] (AsyncStatsGather.result) -> ([world * n, A], [world * n]), ranks in order."""
    a = visits.shape[-1]
    n = visits.shape[0] // (world * wave)
    return (visits.reshape(world, wave, n, a)[:, position].reshape(world * n, a),
            values.reshape(world, wave, n)[:, position].reshape(world * n))


def gather_root_stats(visits, values, group=None):
    """all_gather of per-rank (visits int32 [n, A], values float32 [n]) -> global ([N, A], [N]) on every
    rank, ranks in order.  Equal shard sizes use one all_gather_into_tensor on a packed buffer;
    ragged shards fall back to all_gather on padded rows.  Works on NCCL (CUDA) and gloo (CPU)."""
    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size(group) == 1:
        return visits, values
    world = dist.get_world_size(group)
    n, a = visits.shape
    packed = torch.empty(n, a + 1, dtype=torch.int32, device=visits.device)
    packed[:, :a] = visits
    packed[:, a] = values.contiguous().view(torch.int32)  # bit-cast: one collective for both
    sizes = torch.tensor([n], dtype=torch.int64, device=visits.device)
    all_sizes = [torch.zeros_like(sizes) for _ in range(world)]
    dist.all_gather(all_sizes, sizes, group=group)
    all_sizes = [int(s.item()) for s in all_sizes]
    if len(set(all_sizes)) == 1:
        out = torch.empty(world * n, a + 1, dtype=torch.int32, device=visits.device)
        dist.all_gather_into_tensor(out, packed, group=group)
    else:
        m = max(all_sizes)
        pad = torch.zeros(m, a + 1, dtype=torch.int32, device=visits.device)
        pad[:n] = packed
        bufs = [torch.empty_like(pad) for _ in range(world)]
        dist.all_gather(bufs, pad, group=group)
        out = torch.cat([b[:k] for b, k in zip(bufs, all_sizes)])
    return out[:, :a].contiguous(), out[:, a].contiguous().view(torch.float32)


def gather_root_stats_equal(visits, values, out_packed, group=None):
    """Sync-free variant for the timed path: equal shard sizes, caller-provided int32 [world*n, A+1]."""
    n, a = visits.shape
    packed = out_packed.new_empty(n, a + 1)
    packed[:, :a] = visits
    packed[:, a] = values.view(torch.int32)
    dist.all_gather_into_tensor(out_packed, packed, group=group)
    return out_packed[:, :a], out_packed[:, a].view(torch.float32)


class AsyncStatsGather:
    """The search's one collective, taken off the compute stream: `submit` packs this rank's root statistics and
    issues the all_gather on a side stream that waits only for the statistics kernel, so the next search's
    `Roots.prepare` and simulations run while NCCL moves the 84 B per tree; `result` makes the current stream wait
    for a ticket.  `depth` gathers can be in flight (one packed/out buffer pair each).  Equal shard sizes."""

    def __init__(self, n_local, actions, device, depth=2, group=None):
        self.group, self.depth = group, int(depth)
        self.world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
        self.n, self.a, self.device = int(n_local), int(actions), device
        self.stream = torch.cuda.Stream(device) if device.type == "cuda" else None
        self.slots = [dict(packed=torch.empty(self.n, self.a + 1, dtype=torch.int32, device=device),
                           out=torch.empty(self.world * self.n, self.a + 1, dtype=torch.int32, device=device),
                           done=torch.cuda.Event() if self.stream is not None else None, used=False)
                      for _ in range(self.depth)]
        self._next = 0

    def submit(self, visits, values):
        i = self._next
        self._next = (i + 1) % self.depth
        s = self.slots[i]
        s["flat"] = False
        if self.stream is None:       # gloo / CPU tensors: nothing to overlap with
            s["packed"][:, :self.a] = visits
            s["packed"][:, self.a] = values.contiguous().view(torch.int32)
            if self.world > 1:
                dist.all_gather_into_tensor(s["out"], s["packed"], group=self.group)
            else:
                s["out"].copy_(s["packed"])
            return i
        cur = torch.cuda.current_stream(self.device)
        if s["used"]:
            cur.wait_event(s["done"])            # the slot's previous gather has been consumed in stream order
        self.stream.wait_stream(cur)             # after the statistics kernel (and nothing later)
        with torch.cuda.stream(self.stream):
            s["packed"][:, :self.a] = visits
            s["packed"][:, self.a] = values.view(torch.int32)
            if self.world > 1:
                dist.all_gather_into_tensor(s["out"], s["packed"], group=self.group)
            else:
                s["out"].copy_(s["packed"])
            s["done"].record(self.stream)
        visits.record_stream(self.stream)
        values.record_stream(self.stream)
        s["used"] = True
        return i

    def submit_flat(self, flat):
        """The same collective without any packing: `flat` is this rank's statistics already laid out as one int32
        buffer [n * A visit counts | n value bit patterns] (SearchPipeline lets hz_trees_root_stats write straight
        into such a buffer), gathered as it is.  Read the result with result(ticket) as usual."""
        i = self._next
        self._next = (i + 1) % self.depth
        s = self.slots[i]
        s["flat"] = True
        if self.stream is None:
            if self.world > 1:
                dist.all_gather_into_tensor(s["out"].view(-1), flat, group=self.group)
            else:
                s["out"].view(-1).copy_(flat)
            return i
        cur = torch.cuda.current_stream(self.device)
        if s["used"]:
            cur.wait_event(s["done"])
        self.stream.wait_stream(cur)
        with torch.cuda.stream(self.stream):
            if self.world > 1:
                dist.all_gather_into_tensor(s["out"].view(-1), flat, group=self.group)
            else:
                s["out"].view(-1).copy_(flat, non_blocking=True)
            s["done"].record(self.stream)
        s["used"] = True                         # `flat` is a persistent buffer of the caller: no record_stream needed
        return i

    def result(self, ticket):
        """(visits int32 [world*n, A], values float32 [world*n]) of a ticket; the current stream waits for it."""
        s = self.slots[ticket]
        if self.stream is not None:
            torch.cuda.current_stream(self.device).wait_event(s["done"])
        if s.get("flat"):      # per rank: [n * A visits | n values]
            blocks = s["out"].view(self.world, self.n * (self.a + 1))
            visits = blocks[:, :self.n * self.a].reshape(self.world * self.n, self.a)
            values = blocks[:, self.n * self.a:].reshape(self.world * self.n).view(torch.float32)
            return visits, values
        return s["out"][:, :self.a], s["out"][:, self.a].view(torch.float32)
