"""Written-down restatement of DINO's weighted kNN classifier (`knn_classifier` in DINO's eval_knn.py, Caron et al.
2021) with a stable tie order, in fp64: the statement knn.py is checked against.

    s_ij   = <q_i, k_j>, or the cosine <q_i, k_j> / (||q_i|| ||k_j||) with normalize
    top-k  = the k largest s_ij of row i by decreasing value, equal values by increasing key index
    probs  = probs[i, c] = sum over the top-k neighbours n of query i with label(n) = c of exp(s_in / T)
    top-1  = the label is the first class of probs[i] sorted by decreasing value, equal values by class index
    top-5  = the label is among the first min(5, k) classes of that order

DINO's recipe itself sorts with torch.topk / Tensor.sort, which leave the order of equal values unspecified; this
restatement fixes it.  Row blocks keep the memory at O(block * N_key)."""
from __future__ import annotations

from typing import Dict, Sequence, Tuple, Union

import torch


def scores(queries: torch.Tensor, keys: torch.Tensor, normalize: bool = False) -> torch.Tensor:
    """fp64 [N_q, N_k] scores (the caller picks the block of queries)."""
    q, k = queries.double(), keys.double()
    if normalize:
        q = q / q.norm(dim=1, keepdim=True).clamp_min(1e-12)
        k = k / k.norm(dim=1, keepdim=True).clamp_min(1e-12)
    return q @ k.t()


def stable_topk(s: torch.Tensor, k: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """The k largest entries of every row of s by decreasing value, ties by increasing column index."""
    srt = torch.sort(s, dim=1, descending=True, stable=True)
    return srt.values[:, :k], srt.indices[:, :k]


def knn_topk_ref(queries: torch.Tensor, keys: torch.Tensor, k: int, normalize: bool = False, block: int = 1024
                 ) -> Tuple[torch.Tensor, torch.Tensor]:
    vals, idx = [], []
    for r0 in range(0, queries.shape[0], block):
        v, i = stable_topk(scores(queries[r0:r0 + block], keys, normalize), k)
        vals.append(v)
        idx.append(i)
    return torch.cat(vals), torch.cat(idx)


def vote(values: torch.Tensor, indices: torch.Tensor, train_labels: torch.Tensor, test_labels: torch.Tensor,
         k: int, T: float, num_classes: int) -> Tuple[int, int]:
    """(top-1 hits, top-5 hits) of the weighted vote over the first k neighbours of every row."""
    lab = train_labels.to(indices.device, torch.int64)[indices[:, :k]]
    w = (values[:, :k].double() / T).exp()
    probs = torch.zeros((values.shape[0], num_classes), dtype=torch.float64, device=values.device)
    probs.scatter_add_(1, lab, w)
    order = torch.sort(probs, dim=1, descending=True, stable=True).indices
    correct = order[:, :min(5, k)] == test_labels.to(order.device, torch.int64).view(-1, 1)
    return int(correct[:, 0].sum()), int(correct.sum())


def knn_classify_ref(train_features: torch.Tensor, train_labels: torch.Tensor, test_features: torch.Tensor,
                     test_labels: torch.Tensor, k: Union[int, Sequence[int]] = 20, T: float = 0.07,
                     num_classes: int = None) -> Dict[str, float]:
    ks = [k] if isinstance(k, int) else list(k)
    c = num_classes if num_classes is not None else int(max(train_labels.max(), test_labels.max())) + 1
    values, indices = knn_topk_ref(test_features, train_features, max(ks), normalize=True)
    out = {}
    n = test_features.shape[0]
    for kk in ks:
        t1, t5 = vote(values, indices, train_labels, test_labels, kk, T, c)
        out[f"knn_top1@{kk}"] = t1 * 100.0 / n
        out[f"knn_top5@{kk}"] = t5 * 100.0 / n
    return out


def dino_knn_classifier(train_features, train_labels, test_features, test_labels, k, T, num_classes=1000,
                        chunk=100):
    """DINO's knn_classifier as written (features already L2-normalised, train_features [N_train, d]), in the dtype
    of the inputs: the baseline recipe that knn.py replaces."""
    top1, top5, total = 0.0, 0.0, 0
    train_features = train_features.t()
    num_test_images, num_chunks = test_labels.shape[0], chunk
    imgs_per_chunk = num_test_images // num_chunks if num_test_images >= num_chunks else num_test_images
    imgs_per_chunk = max(imgs_per_chunk, 1)
    retrieval_one_hot = torch.zeros(k, num_classes, dtype=train_features.dtype, device=train_features.device)
    for idx in range(0, num_test_images, imgs_per_chunk):
        features = test_features[idx:min((idx + imgs_per_chunk), num_test_images), :]
        targets = test_labels[idx:min((idx + imgs_per_chunk), num_test_images)]
        batch_size = targets.shape[0]
        similarity = torch.mm(features, train_features)
        distances, indices = similarity.topk(k, largest=True, sorted=True)
        candidates = train_labels.view(1, -1).expand(batch_size, -1)
        retrieved_neighbors = torch.gather(candidates, 1, indices)
        retrieval_one_hot.resize_(batch_size * k, num_classes).zero_()
        retrieval_one_hot.scatter_(1, retrieved_neighbors.view(-1, 1), 1)
        distances_transform = distances.clone().div_(T).exp_()
        probs = torch.sum(torch.mul(retrieval_one_hot.view(batch_size, -1, num_classes),
                                    distances_transform.view(batch_size, -1, 1)), 1)
        _, predictions = probs.sort(1, True)
        correct = predictions.eq(targets.data.view(-1, 1))
        top1 = top1 + correct.narrow(1, 0, 1).sum().item()
        top5 = top5 + correct.narrow(1, 0, min(5, k)).sum().item()
        total += targets.size(0)
    return top1 * 100.0 / total, top5 * 100.0 / total
