"""Specification of det_roi_sample_proposals (csrc/roi_sample.cu) for one image: the labels are the CPU oracle's
roi_label_proposals, the counts its subsample_counts, and the selection keeps each class's smallest hash keys -- numpy
uint32 restatements of mix32 / sample_key / image_seed of csrc/assign.cuh."""
import numpy as np
import torch

from oracle import ref_torch as R

M32 = np.uint64(0xFFFFFFFF)


def mix32(h):
    h = np.asarray(h, dtype=np.uint64) & M32
    h ^= h >> np.uint64(16)
    h = (h * np.uint64(0x7FEB352D)) & M32
    h ^= h >> np.uint64(15)
    h = (h * np.uint64(0x846CA68B)) & M32
    h ^= h >> np.uint64(16)
    return h


def image_seed(seed: int, img: int) -> int:
    seed &= (1 << 64) - 1
    inner = mix32(((seed >> 32) + 0x632BE5AB * (img + 1)) & 0xFFFFFFFF)
    return int(mix32(np.uint64(seed & 0xFFFFFFFF) ^ inner))


def sample_key(img_seed: int, j):
    j = np.asarray(j, dtype=np.uint64)
    return mix32((j * np.uint64(0x9E3779B1) + np.uint64(img_seed)) & M32)


def sample_image(props, gt, gt_classes, num_classes, batch_size_per_image, positive_fraction, seed, img,
                 thresholds=(0.5,), labels=(0, 1), allow_low_quality=False, append_gt=True):
    """One image's rows: dict of boxes (S',4), gt_classes, gt_boxes, matched (int32, -1 without gt), src (int32) with
    S' = count, foreground first, then background, each in ascending candidate index; plus count and num_fg."""
    props = props.reshape(-1, 4).float()
    gt = gt.reshape(-1, 4).float()
    allp, midx, _, cls = R.roi_label_proposals(props, gt, gt_classes.long(), num_classes, thresholds, labels,
                                               allow_low_quality, append_gt)
    fg = ((cls != -1) & (cls != num_classes)).numpy()
    bg = (cls == num_classes).numpy()
    want_pos, want_neg = R.subsample_counts(int(fg.sum()), int(bg.sum()), batch_size_per_image, positive_fraction)
    keys = sample_key(image_seed(seed, img), np.arange(allp.shape[0]))

    def keep(mask, want):
        idx = np.nonzero(mask)[0]
        return np.sort(idx[np.argsort(keys[idx], kind="stable")[:want]])

    src = torch.from_numpy(np.concatenate([keep(fg, want_pos), keep(bg, want_neg)]).astype(np.int64))
    has_gt = gt.shape[0] > 0
    return {"boxes": allp[src], "gt_classes": cls[src],
            "gt_boxes": gt[midx[src]] if has_gt else allp[src],
            "matched": (midx[src] if has_gt else torch.full_like(src, -1)).to(torch.int32),
            "src": src.to(torch.int32), "count": want_pos + want_neg, "num_fg": want_pos}
