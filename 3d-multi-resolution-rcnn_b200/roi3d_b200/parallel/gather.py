"""Multi-GPU plumbing of the RoI path: volumes are independent, so they are sharded round-robin over ranks
(the reference's `range(rank, len(dataset), world_size)`, mmdet/core/evaluation/eval_hooks.py:118) with NO
collective on the data path.  The only exchange is assembling per-volume detections for evaluation, which the
reference does through pickle files on disk plus barriers (eval_hooks.py:134-149, boxes and segm results); here it is
one padded all_gather over NCCL (gloo in the CPU tests), plus one for the masks when they travel along."""
import torch
import torch.distributed as dist


def shard_indices(n_items, rank=None, world_size=None):
    """Indices of the volumes this rank owns."""
    if rank is None:
        rank = dist.get_rank() if dist.is_available() and dist.is_initialized() else 0
    if world_size is None:
        world_size = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
    return list(range(rank, n_items, world_size))


_HEADER_CAP = 256   # volumes a rank announces per round (a rank with more takes several rounds)


def gather_detections(local_dets, local_labels, local_ids, group=None, local_masks=None):
    """All-gather variable-length detections.

    local_dets: list of [n_i, 7] fp32 tensors (one per local volume), local_labels: list of [n_i] int64,
    local_ids: list of global volume ids.  Returns {volume_id: (dets, labels)} on every rank.
    Per round of up to 256 local volumes: one small all_gather of a fixed-size header (volume ids + counts), ONE host
    read of it, then one padded payload all_gather (<= 64 KB per volume -> latency bound).  No per-element host reads.

    local_masks (optional, given on every rank or on none): per local volume the output of
    `models.mask_heads.paste_masks_device`, (boxes int32 [n_i, 6], offsets int64 [n_i + 1], flat uint8 masks, labels).
    Then the header also carries each volume's mask bytes, one padded uint8 all_gather per round carries boxes, offsets
    and masks, and the result is {volume_id: (dets, labels, (boxes, offsets, flat_masks))}.
    """
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        if local_masks is None:
            return {i: (d, l) for i, d, l in zip(local_ids, local_dets, local_labels)}
        return {i: (d, l, tuple(m[:3])) for i, d, l, m in zip(local_ids, local_dets, local_labels, local_masks)}
    world = dist.get_world_size(group)
    dev = local_dets[0].device if local_dets else torch.device('cpu')
    if dist.get_backend(group) == 'nccl' and dev.type != 'cuda':
        dev = torch.device('cuda', torch.cuda.current_device())
    cols = 2 if local_masks is None else 3
    out = {}
    start = 0
    while True:
        ids = local_ids[start:start + _HEADER_CAP]
        dets = local_dets[start:start + _HEADER_CAP]
        labels = local_labels[start:start + _HEADER_CAP]
        masks = None if local_masks is None else local_masks[start:start + _HEADER_CAP]
        more = 1 if start + _HEADER_CAP < len(local_dets) else 0
        # header: row 0 = (volumes in this round, more rounds to come), rows 1.. = (volume id, detections[, mask bytes])
        head_h = torch.full((_HEADER_CAP + 1, cols), -1, dtype=torch.int64)
        head_h[0, 0], head_h[0, 1] = len(dets), more
        for j, (i, d) in enumerate(zip(ids, dets)):
            head_h[1 + j, 0], head_h[1 + j, 1] = int(i), d.shape[0]
            if masks is not None:
                head_h[1 + j, 2] = masks[j][2].numel()
        head = head_h.to(dev)
        heads = [torch.empty_like(head) for _ in range(world)]
        dist.all_gather(heads, head, group=group)
        heads_h = torch.stack(heads).cpu().tolist()           # the one host read of the round
        max_vol = max(h[0][0] for h in heads_h)
        max_n = max([row[1] for h in heads_h for row in h[1:1 + h[0][0]]] + [0])
        if max_vol > 0:
            payload = torch.zeros((max_vol, max(max_n, 1), 8), dtype=torch.float32, device=dev)
            for j, (d, l) in enumerate(zip(dets, labels)):
                n = d.shape[0]
                if n:
                    payload[j, :n, :7] = d.to(dev)
                    payload[j, :n, 7] = l.to(dev).to(torch.float32)
            all_payload = [torch.empty_like(payload) for _ in range(world)]
            dist.all_gather(all_payload, payload, group=group)
            all_mpay = None
            if masks is not None:
                all_mpay = _gather_masks(masks, heads_h, max_vol, dev, world, group)
            for r, (h, p) in enumerate(zip(heads_h, all_payload)):
                for j in range(h[0][0]):
                    vid, n = h[1 + j][:2]
                    out[vid] = (p[j, :n, :7].clone(), p[j, :n, 7].to(torch.int64))
                    if all_mpay is not None:
                        out[vid] += (_unpack_masks(all_mpay[r][j], n, h[1 + j][2]),)
        if not any(h[0][1] for h in heads_h):
            break
        start += _HEADER_CAP
    return out


def _mask_record_bytes(n, mask_bytes):
    """boxes int32 [n, 6], offsets int64 [n + 1], then the masks; rounded up to 8 bytes so that rows stay aligned."""
    return (24 * n + 8 * (n + 1) + mask_bytes + 7) // 8 * 8


def _gather_masks(masks, heads_h, max_vol, dev, world, group):
    width = max(_mask_record_bytes(row[1], row[2]) for h in heads_h for row in h[1:1 + h[0][0]])
    mpay = torch.zeros((max_vol, width), dtype=torch.uint8, device=dev)
    for j, m in enumerate(masks):
        boxes, offsets, flat = m[0], m[1], m[2]
        n, nb = boxes.shape[0], flat.numel()
        mpay[j, :24 * n] = boxes.to(dev, torch.int32).contiguous().view(torch.uint8).reshape(-1)
        mpay[j, 24 * n:24 * n + 8 * (n + 1)] = offsets.to(dev, torch.int64).contiguous().view(torch.uint8).reshape(-1)
        mpay[j, 32 * n + 8:32 * n + 8 + nb] = flat.to(dev).reshape(-1)
    all_mpay = [torch.empty_like(mpay) for _ in range(world)]
    dist.all_gather(all_mpay, mpay, group=group)
    return all_mpay


def _unpack_masks(row, n, mask_bytes):
    boxes = row[:24 * n].clone().view(torch.int32).reshape(n, 6)
    offsets = row[24 * n:32 * n + 8].clone().view(torch.int64)
    return boxes, offsets, row[32 * n + 8:32 * n + 8 + mask_bytes].clone()
