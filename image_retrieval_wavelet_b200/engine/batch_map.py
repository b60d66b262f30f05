"""Mirror of ``/root/reference/main/engine/batch_map.py`` (in-training self-retrieval mAP proxy, :9-36, and the fixed
fast-evaluation subset, :39-91).

In training mode the reference feeds *raw logits* here (``multi_dino_attention.py:750`` only applies ``sign`` in eval
mode), which makes its "Hamming distance" a real-valued proxy, ``0.5 * (B - q @ r.T)`` in float32.
``build_batch_map_calculator(..., on_nonbinary=...)`` picks how logits are ranked:

* ``'sign'`` (default): binarise with bit = logit > 0 and rank by the packed Hamming distance — the mAP the codes would
  have after ``sign()``, a documented deviation from the reference (DESIGN.md §1);
* ``'real'``: rank by the reference's float32 distance (``hamming.real_hamming_map``), so ``compute_batch_map`` on raw
  logits reports the reference's number; batches of exact +-1 codes still take the packed path.
"""
import random

import torch

from .accuracy_calculator import CustomCalculator
from .make_subset import make_subset


def build_batch_map_calculator(distance_metric, device, on_nonbinary="sign"):
    metric_name = "maphashing" if distance_metric == "hamming" else "map"
    calculator = CustomCalculator(exclude=["NMI", "AMI"], k="max_bin_count", with_faiss=False,
                                  distance_metric=distance_metric, device=device, on_nonbinary=on_nonbinary)
    return calculator, metric_name


def compute_batch_map(calculator, metric_name, embeddings, labels):
    with torch.no_grad():
        embeddings = embeddings.detach()
        if labels.ndim == 2 and labels.size(1) == 1:
            labels = labels.view(-1)
        result = calculator.get_accuracy(query=embeddings, query_labels=labels, reference=embeddings,
                                         reference_labels=labels, embeddings_come_from_same_source=True,
                                         include=[metric_name])
    return result[metric_name]


def build_fast_eval_subset(dataset, size, min_per_class=2, seed=0):
    """batch_map.py:39-91 — fixed, stratified self-retrieval subsample of ``dataset``, built once so that it can be
    re-evaluated cheaply and consistently across epochs.  Groups by ``dataset.instance_dict`` ({class / tag index: [image
    indices]}; an image with several active tags sits in several groups, so the selection is de-duplicated as it goes)."""
    rng = random.Random(seed)
    if not hasattr(dataset, "instance_dict"):
        raise AttributeError(
            f"{type(dataset).__name__} has no `instance_dict` -- build_fast_eval_subset needs {{class_or_tag_idx: [image_indices]}} "
            "grouping (see get_instance_dict() on VOC2012Hashing / MIRFlickrHashing for the expected shape).")
    eligible_groups = [idx_list for idx_list in dataset.instance_dict.values() if len(idx_list) >= min_per_class]
    rng.shuffle(eligible_groups)
    selected = []
    seen = set()
    for idx_list in eligible_groups:
        if len(selected) >= size:
            break
        for idx in idx_list:
            if idx not in seen:
                seen.add(idx)
                selected.append(idx)
    selected = selected[:size]
    if not selected:
        raise ValueError(
            f"build_fast_eval_subset found no eligible groups (>= {min_per_class} members) in {type(dataset).__name__}.instance_dict -- "
            "fast_eval_freq should be disabled (-1) for this dataset rather than silently evaluating on an empty subset.")
    subset = make_subset(dataset, selected)
    if hasattr(subset, "_at_R"):
        del subset._at_R
    return subset
