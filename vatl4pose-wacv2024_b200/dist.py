"""Multi-GPU plumbing of the query pass: one process per GPU, torch.distributed for the
rendezvous and the bulk collectives (NCCL over NVLink on GPUs, gloo in the CPU tests), and a
library-owned NCCL communicator for the per-round candidate exchange inside the core-set loop.

Sharding (SURVEY.md §8e): rank r owns the contiguous range [r*n/G, (r+1)*n/G) of the id-sorted
pool.  Heat maps never leave their rank except for one halo frame per side; pooled features are
all-gathered once (1 M x 2048 fp32 = 8.2 GB, fits every GPU) so that the greedy loop only
exchanges one small candidate block per round.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch
import torch.distributed as td

from . import _lib


def shard_range(n: int, rank: int, world: int) -> tuple[int, int]:
    """Contiguous, balanced range of rank `rank` (sizes differ by at most one)."""
    base, rem = divmod(int(n), int(world))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def shard_sizes(n: int, world: int) -> list[int]:
    return [shard_range(n, r, world)[1] - shard_range(n, r, world)[0] for r in range(world)]


# dtypes exchange_halo moves (heat maps: the first three); a dtype code is its index here
_HALO_DTYPES = (torch.float32, torch.float16, torch.bfloat16, torch.float64, torch.int64, torch.int32, torch.int16,
                torch.int8, torch.uint8, torch.bool)


def _agree_dtype(t: torch.Tensor, what: str, group=None):
    """Raise VatlqError on every rank unless every rank's t has the same dtype (one MIN all-reduce on t's device:
    {min code, min -code}, and min == max iff all agree)."""
    code = _HALO_DTYPES.index(t.dtype) if t.dtype in _HALO_DTYPES else len(_HALO_DTYPES)
    mm = torch.tensor([code, -code], dtype=torch.int64, device=t.device)
    td.all_reduce(mm, op=td.ReduceOp.MIN, group=group)
    lo_code, hi_code = int(mm[0].item()), -int(mm[1].item())
    if lo_code != hi_code or code == len(_HALO_DTYPES):
        names = [str(d) for d in _HALO_DTYPES] + ["an unsupported dtype"]
        raise _lib.VatlqError(f"{what}: the ranks hold {'frames' if what == 'exchange_halo' else 'rows'} of different "
                              f"dtypes ({names[lo_code]} .. {names[hi_code]}); every rank must hold the same dtype")


def exchange_halo(first: torch.Tensor | None, last: torch.Tensor | None, rank: int, world: int, group=None):
    """Send this rank's first frame to rank-1 and last frame to rank+1; return
    (halo_prev, halo_next): the frame before / after the local range (None at the pool ends).
    Frames are one (J,h,w) tensor = 208 896 B at the reference shape (104 448 B in fp16 / bf16).  Every rank
    must own at least one frame (shard_range guarantees it for n >= world); an empty shard raises.  The ranks
    first agree on the frames' dtype (one MIN all-reduce on the frames' device): a mismatch raises VatlqError on
    every rank instead of posting sends and receives of different sizes."""
    if world == 1:
        return None, None
    like = first if first is not None else last
    if like is None:
        raise _lib.VatlqError("exchange_halo: an empty shard is not supported (shard_range never produces one "
                              "for n >= world); give every rank at least one frame")
    # every rank must hold one heat-map dtype, or the sends and receives below would not match
    _agree_dtype(like, "exchange_halo", group)
    halo_prev = torch.empty_like(like) if rank > 0 else None
    halo_next = torch.empty_like(like) if rank < world - 1 else None
    ops_ = []
    if rank > 0:
        ops_.append(td.P2POp(td.irecv, halo_prev, _peer(rank - 1, group), group))
        ops_.append(td.P2POp(td.isend, first.contiguous(), _peer(rank - 1, group), group))
    if rank < world - 1:
        ops_.append(td.P2POp(td.isend, last.contiguous(), _peer(rank + 1, group), group))
        ops_.append(td.P2POp(td.irecv, halo_next, _peer(rank + 1, group), group))
    for req in td.batch_isend_irecv(ops_):
        req.wait()
    return halo_prev, halo_next


def _peer(group_rank: int, group):
    return group_rank if group is None else td.get_global_rank(group, group_rank)


def allgather_rows(local: torch.Tensor, n: int, world: int, group=None) -> torch.Tensor:
    """All-gather row shards of unequal length (shard_range layout) into one (n, ...) tensor."""
    sizes = shard_sizes(n, world)
    out = torch.empty((n,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    if world == 1:
        out.copy_(local)
        return out
    if len(set(sizes)) == 1:
        td.all_gather_into_tensor(out, local.contiguous(), group=group)
        return out
    # ragged shards: pad every shard to the longest one, gather, drop the padding
    mx = max(sizes)
    pad = torch.zeros((mx,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    pad[:local.shape[0]] = local
    buf = torch.empty((world * mx,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    td.all_gather_into_tensor(buf, pad, group=group)
    at = 0
    for r, sz in enumerate(sizes):
        out[at:at + sz] = buf[r * mx:r * mx + sz]
        at += sz
    return out


class Comm:
    """Library-owned NCCL communicator (vatlq_comm_*), bootstrapped through torch.distributed."""

    def __init__(self, group=None, use_p2p: bool = True):
        self.rank = td.get_rank(group)
        self.world = td.get_world_size(group)
        self.handle = None
        self.p2p = False
        if self.world == 1:
            return
        L = _lib.lib()
        buf = (C.c_char * 128)()
        if self.rank == 0:
            _lib.check(L.vatlq_comm_unique_id(C.cast(buf, C.c_void_p)), "vatlq_comm_unique_id")
        box = [bytes(buf.raw)]
        td.broadcast_object_list(box, src=_peer(0, group), group=group)
        uid = (C.c_char * 128).from_buffer_copy(box[0])
        out = C.c_void_p()
        _lib.check(L.vatlq_comm_init(C.cast(uid, C.c_void_p), self.rank, self.world, C.byref(out)), "vatlq_comm_init")
        self.handle = out.value
        # peer-memory mailboxes (NVLink): exchange the IPC handles; fall back to NCCL if a peer cannot be mapped
        self.p2p = False
        if use_p2p:
            hb = (C.c_char * 64)()
            _lib.check(L.vatlq_comm_mailbox_handle(C.c_void_p(self.handle), C.cast(hb, C.c_void_p)), "vatlq_comm_mailbox_handle")
            allh = [None] * self.world
            td.all_gather_object(allh, bytes(hb.raw), group=group)
            blob = (C.c_char * (64 * self.world)).from_buffer_copy(b"".join(allh))
            rc = L.vatlq_comm_attach(C.c_void_p(self.handle), C.cast(blob, C.c_void_p), self.world)
            ok = torch.tensor([1 if rc == 0 else 0], device="cuda")
            td.all_reduce(ok, op=td.ReduceOp.MIN, group=group)
            if int(ok.item()) == 1:
                self.p2p = True
            elif rc == 0:
                raise _lib.VatlqError("peer-memory attach succeeded here but failed on another rank")
            else:
                _lib.check(rc, "vatlq_comm_attach")

    def close(self):
        if self.handle:
            _lib.lib().vatlq_comm_destroy(C.c_void_p(self.handle))
            self.handle = None


def distributed_query(H_local, boxes_local, is_prev_local, is_next_local, X_local, ae_weights, labeled_global,
                      n: int, k: int, moks: float = 0.0, lam: float = 0.01, uncertainty: str = "THC+WPU",
                      thc_vs_wpu: str = "const", rule: str = "w_unc", batch: int = 16, comm: Comm | None = None,
                      group=None, first_pick: int = -1, representativeness: str = "None", filter: str = "Coreset",
                      w_unc: float = 1.0):
    """One query over a pool sharded across the ranks of `group` (one process per GPU).
    Every rank passes its slice of the pool and gets the same global pick list back.  Heat-map shards may be
    fp32, fp16 or bf16 (the same dtype on every rank; the picks equal those of the fp32 upcast), and so may the
    embedding shards X_local for representativeness "Influence" and every filter: Influence reads each rank's
    shard as it is, the filters gather the shards and select on them as they are, and the scores and picks equal
    those of the fp32 upcast.  Every rank must hold X_local in one dtype (checked once, on every rank, before the
    first step that reads it).
    uncertainty: any accelerated name (THC*, WPU*, THC+WPU, HP, TPC, Entropy, MPE, Margin, None);
    representativeness: "None" or "Influence" (ActiveLearning.py:467-477); filter: "Coreset" (:609-614),
    "None" (top-k, :533-534), "Diversity" (:581-590), "K-Means" (:593-608) or "weighted" (:553-580; w_unc = cfg.VAL.W_UNC;
    the assignment step of Lloyd is sharded by rows, seeding and the M step run replicated).  With at most one
    unlabelled item every filter returns the score-ordered top k of the unlabelled items, like the reference
    (:533-534, 541-542).  Scoring is sharded (halo frame / halo coordinates for
    THC / TPC, MIN all-reduces for the normalisations, a SUM all-reduce of the cosine column sums for
    Influence); the fused scores are all-gathered (8 B per item) and the filter runs replicated (query.select)."""
    from . import ops
    from .query import FILTERS, QueryPass, QueryResult, influence, select, unlabelled_mask
    if representativeness not in ("None", "Influence"):
        raise ValueError("Representativeness type is not supported by distributed_query")
    if filter not in FILTERS:
        raise ValueError("Filter type is not supported by distributed_query")
    rank, world = td.get_rank(group), td.get_world_size(group)
    lo, hi = shard_range(n, rank, world)
    dev = X_local.device
    qp = QueryPass(hi - lo, dev, ae_weights=ae_weights, uncertainty=uncertainty)
    if isinstance(H_local, (list, tuple)):     # (pos, tensor) segments in pool order
        first = H_local[0][1][0] if H_local else None
        last = H_local[-1][1][-1] if H_local else None
    else:
        first = H_local[0] if hi > lo else None
        last = H_local[-1] if hi > lo else None
    hp, hn = exchange_halo(first, last, rank, world, group)
    qp.score_pool(H_local, boxes_local, is_prev_local, is_next_local, halo_prev=hp, halo_next=hn)
    lab = np.asarray(list(labeled_global), dtype=np.int64)
    unl = unlabelled_mask(n, lab, dev)
    # (group=None means the default group to torch.distributed but "single GPU" to QueryPass.fuse)
    fuse_group = (group if group is not None else td.group.WORLD) if world > 1 else None
    n_unl = n - lab.size
    # every rank must hold one embedding dtype: the all-gather of the filters needs one row size, and Influence's
    # column sums are only the upcast's when every shard is read the same way (filter "None" reads no X)
    if world > 1 and (representativeness == "Influence" or filter != "None"):
        _agree_dtype(X_local, "distributed_query", group)
    score_local = qp.fuse(unl[lo:hi], thc_vs_wpu, labeled_ratio=lab.size / max(n, 1), group=fuse_group,
                          n_unlabeled_global=n_unl)
    if representativeness == "Influence" and n_unl > 1:                      # (:467-477, 517-526)
        infl = influence(X_local, unl[lo:hi], group=fuse_group)
        score_local = ops.blend_scores(score_local, infl, qp.combine_weight, unl[lo:hi]) if uncertainty != "None" else infl
    score = allgather_rows(score_local, n, world, group)

    def gather_X():
        return allgather_rows(X_local, n, world, group)
    picks, _, st = select(score, unl, gather_X, k, filter, labeled=lab, moks=moks, lam=lam, rule=rule,
                          first_pick=first_pick, batch=batch, comm=comm.handle if comm is not None else None,
                          row_range=(lo, hi) if world > 1 else None, w_unc=w_unc, combine_weight=qp.combine_weight,
                          group=fuse_group)
    return QueryResult(picks=picks, thc=qp.thc, wpu=qp.wpu, peak_mean=qp.peak_mean, kpts=qp.kpts, unc=score,
                       combine_weight=qp.combine_weight, stats=st)
