# -*- coding: utf-8 -*-
"""Multi-GPU keyphrase table and keyphrase graph: documents shard over ranks.

The reference has no distributed code (SURVEY 2.1); its unit of independence is the document
(one AST per text, east/relevance.py:41-47).  One process per GPU (torch.distributed, NCCL over
NVLink on the GPU box, gloo in CPU tests): every rank indexes and scores a contiguous range of
documents against the replicated keyphrases.

Table.  The doc-major [D_r, K] float64 slices concatenate into the [D, K] table (SURVEY 5.8).  Two ways to
join them:
  * fused (default on NCCL/CUDA when torch symmetric memory is available): the gathered table lives in
    symmetric memory; every rank passes the addresses of its rows in the other ranks' tables to
    east_table_dev_gather and the CTA that scores a document stores its row to all of them (NVLink peer
    stores) -- the all-gather happens inside the scoring kernel, row by row; one barrier ends the step;
  * one all_gather_into_tensor of the slices (padded to a common height) -- gloo, ragged batches, no
    symmetric memory.
Graph.  Co-occurrence counts are additive over documents: every rank indexes its own documents and counts
C_r = B_r B_r^T of their relevance bytes on the tensor cores (east_graph_dev: the scoring kernel writes the bytes, no
score table is formed), and ONE all_reduce(int32 sum) of the K x K counts joins them (east/applications.py:111-147;
SURVEY 5.8).  There is no other exchange on the path.
"""
import numpy as np


def partition_documents(sizes, world_size):
    """Contiguous document ranges balanced by total size (code points).

    Returns [(begin, end)] * world_size; ranges may be empty when there are fewer documents
    than ranks.  Deterministic, so every rank computes the same partition."""
    sizes = np.asarray(sizes, dtype=np.int64)
    n = len(sizes)
    bounds = [0]
    if n:
        csum = np.cumsum(sizes)
        total = int(csum[-1])
        for r in range(1, world_size):
            target = total * r / float(world_size)
            cut = int(np.searchsorted(csum, target, side="left"))
            # put the boundary document where the imbalance is smaller
            if cut < n and cut >= bounds[-1]:
                before = csum[cut - 1] if cut > 0 else 0
                if abs(csum[cut] - target) < abs(before - target):
                    cut += 1
            bounds.append(min(max(cut, bounds[-1]), n))
    else:
        bounds += [0] * (world_size - 1)
    bounds.append(n)
    return [(bounds[r], bounds[r + 1]) for r in range(world_size)]


def gather_score_slices(local_scores, ranges, group=None):
    """All-gather the per-rank [D_r, K] slices into the full [D, K] table (on every rank).

    local_scores: torch float64 tensor [D_r, K] on this rank's device (CUDA for NCCL, CPU for gloo).
    ranges: the partition from partition_documents (same on all ranks)."""
    import torch
    import torch.distributed as dist

    world = dist.get_world_size(group)
    K = int(local_scores.shape[1])
    heights = [e - b for b, e in ranges]
    max_h = max(heights) if heights else 0
    if max_h == 0:
        return local_scores.new_zeros((0, K))
    padded = local_scores.new_zeros((max_h, K))
    padded[: local_scores.shape[0]] = local_scores
    gathered = local_scores.new_empty((world * max_h, K))
    dist.all_gather_into_tensor(gathered, padded, group=group)
    if all(h == max_h for h in heights):
        return gathered
    return torch.cat([gathered[r * max_h: r * max_h + heights[r]] for r in range(world)], dim=0)


class SymmetricTable(object):
    """A [rows, K] float64 table in torch symmetric memory: every rank's copy is mapped into every other rank's
    address space, so a kernel of rank r can store rows straight into the tables of its peers."""

    def __init__(self, rows, K, device, group=None):
        import torch
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm_mem
        self.group = group if group is not None else dist.group.WORLD
        self.rank = dist.get_rank(self.group)
        self.world = dist.get_world_size(self.group)
        self.K = int(K)
        self.tensor = symm_mem.empty((max(int(rows), 1), self.K), dtype=torch.float64, device=torch.device("cuda", device))
        self.handle = symm_mem.rendezvous(self.tensor, self.group)
        self.tensor = self.tensor[:rows]
        self.buffer_ptrs = [int(p) for p in self.handle.buffer_ptrs]

    def peer_rows(self, first_row):
        """Addresses of row `first_row` in the tables of the OTHER ranks (what east_table_dev_gather takes)."""
        off = int(first_row) * self.K * 8
        return [self.buffer_ptrs[r] + off for r in range(self.world) if r != self.rank]

    def own_rows(self, first_row):
        return self.buffer_ptrs[self.rank] + int(first_row) * self.K * 8

    def barrier(self):
        """Every rank's stores (fenced system-wide by the kernels that made them) are visible once all ranks
        have passed this barrier; it is queued on the current stream."""
        self.handle.barrier(channel=0)


def symmetric_memory_available(group=None):
    """True when the process group runs on NCCL/CUDA and torch can allocate + rendezvous symmetric memory."""
    try:
        import torch
        import torch.distributed as dist
        import torch.distributed._symmetric_memory  # noqa: F401
        return (dist.is_initialized() and dist.get_backend(group) == "nccl" and torch.cuda.is_available()
                and dist.get_world_size(group) <= 16)
    except Exception:  # noqa: BLE001
        return False


def _pack_local(texts):
    """Host preprocessing + packing of this rank's texts: (uint32 text, doc_off, doc_m, batches of document numbers)."""
    from east import utils
    from east.asts import utils as asts_utils
    from east.relevance import plan_batches
    cols = [utils.text_to_strings_collection(t) for t in texts]
    packed = [asts_utils.pack_strings_collection(c) for c in cols]
    return cols, packed, plan_batches([len(p) for p in packed])


def _upload_batch(packed, cols, docs, dev):
    """One device batch of _pack_local's documents: (its packed text concatenated on `dev`, doc_off, doc_m)."""
    import torch
    doc_off = np.zeros(len(docs) + 1, dtype=np.int64)
    np.cumsum([len(packed[j]) for j in docs], out=doc_off[1:])
    text = np.ascontiguousarray(np.concatenate([packed[j] for j in docs]) if len(docs) > 1 else packed[docs[0]], dtype=np.uint32)
    return torch.from_numpy(text.view(np.int32)).to(dev), doc_off, [len(cols[j]) for j in docs]


def relevance_table_sharded(texts, prepared_keyphrases, normalized=True, device=None, group=None, fused_gather=None,
                            return_local=False, synonimizer=None):
    """[D, K] float64 score table of all texts x keyphrases, computed by all ranks together.

    texts: list of raw texts (same list on every rank).  Each rank preprocesses, packs, indexes and scores only
    its own range on its own GPU (east_table_dev: one engine call builds and scores a batch); returns the gathered
    table as a torch tensor on that GPU (with return_local: also this rank's (begin, end) rows).
    synonimizer: the synonym table of ASTRelevanceMeasure.relevance_table(prepared_keyphrases, synonimizer) -- the best
    variant of each keyphrase, always normalized (east_table_groups_dev), with the same two ways to gather."""
    import torch
    import torch.distributed as dist

    from east import _capi

    rank = dist.get_rank(group)
    world = dist.get_world_size(group)
    if device is None:
        device = torch.cuda.current_device()
    dev = torch.device("cuda", device)
    ranges = partition_documents([len(t) for t in texts], world)
    begin, end = ranges[rank]
    group_off = None
    if synonimizer:
        codes, off, group_off = _capi.pack_variant_groups(prepared_keyphrases, synonimizer.get_synonyms())
    else:
        codes, off = _capi.pack_keyphrases(prepared_keyphrases)
    K = len(prepared_keyphrases)   # columns: one per keyphrase (with synonyms: one per group of variants)
    D = len(texts)
    cols, packed, batches = _pack_local(texts[begin:end]) if end > begin else ([], [], [])
    # the fused gather writes the rows of ONE batch of consecutive documents; ragged collections (small and large
    # documents apart, several device batches) take the all-gather.  All ranks must agree: the choice is all-reduced.
    want_fused = (fused_gather if fused_gather is not None else True) and symmetric_memory_available(group)
    mine = 1 if (want_fused and len(batches) <= 1) else 0
    flag = torch.tensor([mine], dtype=torch.int32, device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
    fused = bool(flag.item())
    stream = torch.cuda.current_stream(dev)
    kp_dev = torch.from_numpy(codes.view(np.int32).copy()).to(dev)

    def score_batch(docs, out_ptr, peer_rows):
        text_dev, doc_off, doc_m = _upload_batch(packed, cols, docs, dev)
        _capi.DeviceIndex.build_dev_and_score(text_dev.data_ptr(), doc_off, doc_m, kp_dev.data_ptr(), codes, off, out_ptr,
                                              normalized, device=device, stream=stream.cuda_stream, peer_rows=peer_rows,
                                              group_off=group_off).close()

    table = None
    if fused:
        # allocation + rendezvous are collective; if they fail anywhere every rank takes the all-gather
        try:
            table = SymmetricTable(D, K, device, group)
        except Exception:  # noqa: BLE001
            table = None
        flag = torch.tensor([1 if table is not None else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
        fused = bool(flag.item())
    if fused:
        if batches:
            score_batch(batches[0], table.own_rows(begin), table.peer_rows(begin))
        table.barrier()
        torch.cuda.synchronize(dev)
        full = table.tensor
        full._east_symmetric = table   # keeps the rendezvous handle alive with the tensor
    else:
        local = torch.empty((end - begin, K), dtype=torch.float64, device=dev)
        for docs in batches:
            if len(batches) == 1:
                score_batch(docs, local.data_ptr(), None)
            else:
                rows = torch.empty((len(docs), K), dtype=torch.float64, device=dev)
                score_batch(docs, rows.data_ptr(), None)
                local[torch.as_tensor(docs, device=dev)] = rows
        full = gather_score_slices(local, ranges, group)
    return (full, (begin, end)) if return_local else full


def cooccurrence_sharded(local_scores, relevance_threshold, device=None, group=None):
    """int32 [K, K] co-occurrence counts of the whole collection (east/applications.py:111-113, 136-147) from
    this rank's [D_r, K] rows of the score table: C_r = B_r B_r^T on the tensor cores, then ONE all_reduce(sum).
    local_scores: torch float64 CUDA tensor (may have zero rows)."""
    import torch
    import torch.distributed as dist

    from east import _capi
    if device is None:
        device = local_scores.device.index
    K = int(local_scores.shape[1])
    C = torch.zeros((K, K), dtype=torch.int32, device=local_scores.device)
    if local_scores.shape[0] > 0:
        S = local_scores.contiguous()
        _capi.cooc_dev(S.data_ptr(), S.shape[0], K, relevance_threshold, C.data_ptr(), device=device,
                       stream=torch.cuda.current_stream(local_scores.device).cuda_stream)
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(C, op=dist.ReduceOp.SUM, group=group)
    return C


def keyphrases_graph_sharded(keyphrases, texts, referral_confidence=0.6, relevance_threshold=0.25, support_threshold=1,
                             normalized=True, device=None, group=None, synonimizer=None):
    """applications.keyphrases_graph computed by all ranks together: the same graph dict on every rank.

    texts: {name: text} (same on every rank); documents shard over the ranks, every rank indexes its own and counts
    its own co-occurrences with one graph call per device batch (east_graph_dev; several batches are summed on the
    device); the K x K counts are all-reduced.  No rank forms a score table.  synonimizer: as in keyphrases_graph."""
    import torch
    import torch.distributed as dist

    from east import _capi
    from east import applications
    from east import utils
    kept = [kp for kp in keyphrases if kp]
    prepared = [utils.prepare_text(kp) for kp in kept]
    text_collection = list(texts.values())
    rank = dist.get_rank(group)
    world = dist.get_world_size(group)
    if device is None:
        device = torch.cuda.current_device()
    dev = torch.device("cuda", device)
    begin, end = partition_documents([len(t) for t in text_collection], world)[rank]
    K = len(prepared)
    cooc = torch.zeros((K, K), dtype=torch.int32, device=dev)
    cols, packed, batches = _pack_local(text_collection[begin:end]) if end > begin and K else ([], [], [])
    if batches:
        group_off = None
        if synonimizer:
            codes, off, group_off = _capi.pack_variant_groups(prepared, synonimizer.get_synonyms())
        else:
            codes, off = _capi.pack_keyphrases(prepared)
        stream = torch.cuda.current_stream(dev)
        kp_dev = torch.from_numpy(codes.view(np.int32).copy()).to(dev)
        part = torch.empty_like(cooc) if len(batches) > 1 else cooc
        for b, docs in enumerate(batches):
            text_dev, doc_off, doc_m = _upload_batch(packed, cols, docs, dev)
            target = cooc if b == 0 else part
            _capi.DeviceIndex.build_dev_and_graph(text_dev.data_ptr(), doc_off, doc_m, kp_dev.data_ptr(), codes, off,
                                                  relevance_threshold, target.data_ptr(), normalized, device=device,
                                                  stream=stream.cuda_stream, group_off=group_off).close()
            if b > 0:
                cooc += part   # int32: exact
    if world > 1:
        dist.all_reduce(cooc, op=dist.ReduceOp.SUM, group=group)
    return applications.graph_from_cooccurrence(keyphrases, kept, cooc.cpu().numpy(), referral_confidence,
                                                relevance_threshold, support_threshold)
