"""Device-resident hand-off from feature extraction to the pseudo-label pass (SURVEY.md 8f, row f4).

The reference moves every batch of backbone outputs to the host (`outputs.data.cpu()`, clustercontrast/evaluators.py:19),
keeps one CPU tensor per file name in an OrderedDict (:46-53) and re-assembles the (N, 2048) matrix with an N-way
`torch.cat` on the host (examples/cluster_contrast_train_usl.py:152-153) -- only for compute_jaccard_distance to upload it
again.  Here the outputs stay where the backbone produced them:

    features, labels = extract_features(model, cluster_loader)           # same call, same return shape
    x = features.matrix([f for f, _, _ in sorted(dataset.train)])        # (N, D) CUDA tensor, one gather kernel
    out = pipeline.pseudo_labels(x, k1, k2, eps)                         # or compute_jaccard_distance(x, ...)

`features` is a DeviceFeatures: an OrderedDict-like view (file name -> (D,) row, CUDA) over ONE device buffer, so code
written against the reference's dict keeps working (`features[f]`, iteration, len).  With one process per GPU each rank
extracts only its contiguous share of the sorted list (`shard_items`) and hands its rows to
`sharded.pseudo_labels(x_local, N=N)`: collective (1) of SURVEY 8(e), the feature all-gather, then moves fp32 rows over
NVLink instead of every rank extracting or uploading all N.

`Evaluator` and `evaluate_all` are the drop-ins of the evaluation entry points (evaluators.py:91-142): the features
stay on the device, the Q x G distance matrix is computed there and scored there, and `rerank=True` re-ranks from the
features (rerank.re_ranking_features, reusing the Q x G block) -- no Q x Q or G x G matrix and no host copy of any
distance matrix.
"""
import time
from collections import OrderedDict

import torch

from . import _lib
from ._lib import call, ptr, stream_ptr


class DeviceFeatures:
    """file name -> feature row, backed by one (capacity, D) CUDA buffer that grows geometrically."""

    def __init__(self, device=None):
        self.device = device
        self._buf = None
        self._rows = OrderedDict()          # name -> row index (insertion order, like the reference's OrderedDict)

    # -- filling -----------------------------------------------------------------------------
    def append_batch(self, names, outputs):
        if not outputs.is_cuda:
            raise RuntimeError("DeviceFeatures keeps CUDA tensors; there is no CPU fallback")
        outputs = outputs.detach().to(torch.float32)
        b, d = outputs.shape
        if len(names) != b:
            raise ValueError("%d names for %d rows" % (len(names), b))
        n0 = len(self._rows)
        if self._buf is None:
            self.device = outputs.device
            self._buf = torch.empty((max(1024, 2 * b), d), dtype=torch.float32, device=self.device)
        if n0 + b > self._buf.shape[0]:
            grown = torch.empty((max(2 * self._buf.shape[0], n0 + b), d), dtype=torch.float32, device=self.device)
            grown[:n0].copy_(self._buf[:n0])
            self._buf = grown
        fresh = [nm for nm in names if nm not in self._rows]
        if len(fresh) == b:
            self._buf[n0:n0 + b].copy_(outputs)                         # device-to-device, no host round trip
            for i, nm in enumerate(names):
                self._rows[nm] = n0 + i
        else:                                                           # a name seen before is overwritten in place
            for i, nm in enumerate(names):
                r = self._rows.get(nm)
                if r is None:
                    r = len(self._rows)
                    self._rows[nm] = r
                self._buf[r].copy_(outputs[i])

    # -- the reference's dict surface ------------------------------------------------------------
    def __len__(self):
        return len(self._rows)

    def __contains__(self, name):
        return name in self._rows

    def __getitem__(self, name):
        return self._buf[self._rows[name]]

    def __iter__(self):
        return iter(self._rows)

    def keys(self):
        return self._rows.keys()

    def values(self):
        return (self._buf[r] for r in self._rows.values())

    def items(self):
        return ((nm, self._buf[r]) for nm, r in self._rows.items())

    # -- hand-off ----------------------------------------------------------------------------
    def matrix(self, names=None):
        """(len(names), D) contiguous CUDA tensor with the rows in the order of `names` (default: insertion order)."""
        n = len(self._rows)
        if n == 0:
            raise RuntimeError("no features were extracted")
        if names is None:
            return self._buf[:n]
        idx = [self._rows[nm] for nm in names]
        if idx == list(range(len(idx))):
            return self._buf[:len(idx)]
        d = self._buf.shape[1]
        with torch.cuda.device(self.device):
            idx_d = torch.tensor(idx, dtype=torch.int64).to(self.device, non_blocking=True)
            out = torch.empty((len(idx), d), dtype=torch.float32, device=self.device)
            if d % 4 == 0:
                call("reid_gather_rows", ptr(self._buf), n, ptr(idx_d), len(idx), d, ptr(out), stream_ptr())
            else:
                out.copy_(self._buf[idx_d])
        return out


def extract_cnn_feature(model, inputs):
    """evaluators.py:16-20 without the `.cpu()`: the outputs stay on the device."""
    inputs = inputs if isinstance(inputs, torch.Tensor) else torch.as_tensor(inputs)
    return model(inputs.cuda()).data


def extract_all_feature(model, inputs):
    """evaluators.py:22-27 without the `.cpu()`."""
    inputs = inputs if isinstance(inputs, torch.Tensor) else torch.as_tensor(inputs)
    outputs, extra_outputs = model(inputs.cuda(), test_all=True)
    return outputs.data, extra_outputs.data


def extract_features(model, data_loader, print_freq=50, extra_features=False):
    """evaluators.py:30-68, same signature and return shape; `features` (and `gan_features`) are DeviceFeatures."""
    model.eval()
    features, labels = DeviceFeatures(), OrderedDict()
    gan_features = DeviceFeatures() if extra_features else None
    end = time.time()
    with torch.no_grad():
        for i, (imgs, fnames, pids, _, _) in enumerate(data_loader):
            if extra_features:
                outputs, extra_outputs = extract_all_feature(model, imgs)
                gan_features.append_batch(list(fnames), extra_outputs)
            else:
                outputs = extract_cnn_feature(model, imgs)
            features.append_batch(list(fnames), outputs)
            for fname, pid in zip(fnames, pids):
                labels[fname] = pid
            if (i + 1) % print_freq == 0:
                print('Extract Features: [{}/{}]\tTime {:.3f}'.format(i + 1, len(data_loader), time.time() - end))
            end = time.time()
    if extra_features:
        return features, gan_features, labels
    return features, labels


def shard_items(sorted_items, group=None, world=None, rank=None):
    """This rank's contiguous share of the sorted training list -- rows [N r / W, N (r + 1) / W), the partition of
    sharded.RowComm -- plus (row_begin, row_end, N).  Build the cluster loader over it, extract, and pass
    `features.matrix(names_of_the_share)` to sharded.pseudo_labels(x_local, N=N)."""
    from .sharded import partition
    if world is None:
        import torch.distributed as dist
        world, rank = dist.get_world_size(group), dist.get_rank(group)
    n = len(sorted_items)
    r0, r1 = partition(n, world, rank)
    return list(sorted_items[r0:r1]), r0, r1, n


def evaluate_all(query_features, gallery_features, distmat, query=None, gallery=None, query_ids=None, gallery_ids=None,
                 query_cams=None, gallery_cams=None, cmc_topk=(1, 5, 10), cmc_flag=False):
    """evaluators.py:91-124.  Returns mAP, or (cmc_scores, mAP) with cmc_flag (the 'market1501' CMC configuration).
    `distmat` may be a CUDA tensor: it is scored where it is."""
    from .evaluation import cmc, mean_ap
    if query is not None and gallery is not None:
        query_ids = [pid for _, pid, _ in query]
        gallery_ids = [pid for _, pid, _ in gallery]
        query_cams = [cam for _, _, cam in query]
        gallery_cams = [cam for _, _, cam in gallery]
    else:
        assert (query_ids is not None and gallery_ids is not None
                and query_cams is not None and gallery_cams is not None)
    mAP = mean_ap(distmat, query_ids, gallery_ids, query_cams, gallery_cams)
    print('Mean AP: {:4.1%}'.format(mAP))
    if not cmc_flag:
        return mAP
    cmc_configs = {
        'market1501': dict(separate_camera_set=False, single_gallery_shot=False, first_match_break=True)}
    cmc_scores = {name: cmc(distmat, query_ids, gallery_ids, query_cams, gallery_cams, **params)
                  for name, params in cmc_configs.items()}
    print('CMC Scores:')
    for k in cmc_topk:
        print('  top-{:<4}{:12.1%}'.format(k, cmc_scores['market1501'][k - 1]))
    return cmc_scores['market1501'], mAP


class Evaluator(object):
    """evaluators.py:127-142 on the device: one gather each for the query and gallery rows of the extracted features,
    the Q x G distances on the device, metrics on the device; rerank=True re-ranks from the features."""

    def __init__(self, model):
        super(Evaluator, self).__init__()
        self.model = model

    def evaluate(self, data_loader, query, gallery, cmc_flag=False, rerank=False):
        from .evaluation import pairwise_distance_device
        from .rerank import _re_ranking_features
        features, _ = extract_features(self.model, data_loader)
        dev = features.device
        with torch.cuda.device(dev), torch.no_grad():
            query_features = features.matrix([f for f, _, _ in query])
            gallery_features = features.matrix([f for f, _, _ in gallery])
            distmat = pairwise_distance_device(query_features, gallery_features)
        results = evaluate_all(query_features, gallery_features, distmat, query=query, gallery=gallery, cmc_flag=cmc_flag)
        if not rerank:
            return results
        print('Applying person re-ranking ...')
        distmat, _ = _re_ranking_features(query_features, gallery_features, q_g_dist=distmat)
        return evaluate_all(query_features, gallery_features, distmat, query=query, gallery=gallery, cmc_flag=cmc_flag)
