"""Multi-GPU plumbing (one process per GPU): template sharding by tmpl_idx, scene sharding and the merge of the
per-rank top-K match lists (SURVEY.md §8e).  The data path has no other collective: every rank builds (or receives) the
scene's feature map and searches its own shard.

Two layers:
  * `Communicator` — the product path: the C ABI's fdcm_comm_* entry points (NCCL all-gather of the k x 32-byte top-K
    buffer on the compute stream + merge kernel on the device, one download; ncclBroadcast of a built map).  The NCCL
    unique id is shipped with torch.distributed (any transport would do).
  * `allgather_topk` / `merge_topk_records` — the same exchange through torch.distributed tensors, kept for CPU (`gloo`)
    tests of the host logic and as the reference the device merge is tested against.
"""
import ctypes as C

import numpy as np
import torch
import torch.distributed as dist

from . import _lib
from ._lib import MATCH_DTYPE, check, lib, ptr


class Communicator:
    """fdcm_comm of this rank.  `Communicator.from_torch()` bootstraps from an initialised torch.distributed group."""

    def __init__(self, unique_id, rank, world, device):
        uid = np.frombuffer(bytes(unique_id), np.uint8).copy()
        assert uid.size == 128
        h = C.c_void_p(0)
        check(lib().fdcm_comm_init(ptr(uid), int(rank), int(world), int(device), C.byref(h)))
        self._h, self.rank, self.world, self.device = h, int(rank), int(world), int(device)

    @staticmethod
    def unique_id():
        uid = np.zeros(128, np.uint8)
        check(lib().fdcm_comm_unique_id(ptr(uid)))
        return uid.tobytes()

    @classmethod
    def from_torch(cls, device, group=None):
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        box = [cls.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0, group=group)
        return cls(box[0], rank, world, device)

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h and lib is not None:   # (module globals are gone when the interpreter shuts down)
            lib().fdcm_comm_destroy(h)

    def shard(self, n_items):
        b, e = C.c_int32(0), C.c_int32(0)
        check(lib().fdcm_comm_shard(int(n_items), self.rank, self.world, C.byref(b), C.byref(e)))
        return b.value, e.value

    def search_topk(self, featuremap, shard, scene, searcher, optimizer, penalty, k, tmpl_idx_base, *, select=None):
        """Search this rank's shard (a TemplateSet) and return the GLOBAL top-k (same on every rank).  select: a
        DistinctMatches without across_templates (the distinct top-k of the whole template set)."""
        from . import _records
        s = None if scene is None else _records(scene)
        p = _lib.SearchParams(searcher.max_tmpl_lines, searcher.max_scene_lines, int(optimizer.batch_size),
                              0 if penalty is None else penalty.kind, 0.0 if penalty is None else float(penalty.tau),
                              int(k), int(tmpl_idx_base), 0, 0.0, 0.0, 0.0, 0.0)
        out = np.zeros(int(k), MATCH_DTYPE)
        n = C.c_int64(0)
        n_scene = _lib.FDCM_SCENE_RESIDENT if s is None else s.shape[0]
        if select is None:
            check(lib().fdcm_comm_search_topk(self._h, featuremap._h, shard._h, ptr(s), n_scene, C.byref(p), ptr(out), int(k), C.byref(n)))
        else:
            sp = select._params()
            check(lib().fdcm_comm_search_select(self._h, featuremap._h, shard._h, ptr(s), n_scene, C.byref(p), C.byref(sp), ptr(out), int(k),
                                                C.byref(n)))
        return out[: n.value].copy()

    def rebuild_broadcast(self, featuremap, scene, root=0):
        """Every rank ends up with the map of `scene`; only `root` runs the build kernels (ncclBroadcast of the planes)."""
        from . import _records
        r = _records(scene)
        check(lib().fdcm_comm_rebuild_broadcast(self._h, featuremap._h, ptr(r), r.shape[0], int(root)))
        featuremap._refresh()


def shard_range(n_items, rank, world):
    """Contiguous, balanced shard [begin, end) of n_items for `rank` of `world`."""
    base, rem = divmod(n_items, world)
    begin = rank * base + min(rank, rem)
    return begin, begin + base + (1 if rank < rem else 0)


def shard_templates(templates, rank, world):
    """Contiguous shard of the template list; returns (templates_of_rank, tmpl_idx_base)."""
    b, e = shard_range(len(templates), rank, world)
    return templates[b:e], b


def shard_scenes(n_scenes, rank, world):
    """Scene s goes to rank s % world (config 5: multi-view batches)."""
    return list(range(rank, n_scenes, world))


def merge_topk_records(per_rank, k):
    """Merge per-rank top-k MATCH_DTYPE arrays: ascending score, ties by (rank order, local order)."""
    allm = np.concatenate([np.asarray(r, MATCH_DTYPE) for r in per_rank]) if per_rank else np.zeros(0, MATCH_DTYPE)
    order = np.argsort(allm["score"], kind="stable")
    return allm[order[:k]]


def allgather_topk(local_topk, k, device=None, group=None):
    """All-gather the ranks' top-k lists (k x 32 B each, padded) and merge them locally on every rank."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    local = np.zeros(k, MATCH_DTYPE)
    n = min(k, len(local_topk))
    local[:n] = local_topk[:n]
    local["score"][n:] = np.inf
    local["tmpl_idx"][n:] = -1
    if world == 1:
        return merge_topk_records([local[:n]], k)
    buf = torch.from_numpy(local.view(np.uint8).copy())
    if device is not None:
        buf = buf.to(device, non_blocking=False)
    out = torch.empty(world * buf.numel(), dtype=torch.uint8, device=buf.device)
    dist.all_gather_into_tensor(out, buf, group=group)
    rec = out.cpu().numpy().view(MATCH_DTYPE).reshape(world, k)
    return merge_topk_records([r[r["tmpl_idx"] >= 0] for r in rec], k)


def broadcast_featuremap(featuremap, src=0, group=None):
    """NCCL-broadcast the planes of `featuremap` from rank `src` into the same-shaped maps of the other ranks
    (alternative to every rank rebuilding the scene's map; SURVEY.md §8e — use whichever measures faster)."""
    ptr, nbytes = featuremap.device_ptr()
    n = nbytes // 4

    class _Blob:
        __cuda_array_interface__ = {"shape": (n,), "typestr": "<f4", "data": (ptr, False), "version": 3}

    t = torch.as_tensor(_Blob(), device=f"cuda:{featuremap.device}")
    dist.broadcast(t, src=src, group=group)
    torch.cuda.synchronize(featuremap.device)
