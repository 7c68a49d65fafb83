"""Oracle: a query's genotypes in a stored model's site order (CPU, plain loops).

TEST INFRASTRUCTURE -- see oracle/__init__.py.  Restates what python -m locator_b200.predict hands the first layer
(loc_pack_sites_mapped / loc_bed_pack_sites_mapped): model site k reads query record src[k] (-1: the query lacks
it); a call whose two alleles are both 0 or 1 gives its count of allele 1, or of allele 0 when flip[k] is set; any
other call (missing, half-missing, an allele index >= 2) and every call of an absent site gives 3.  A .bed query is
its GT cube (oracle/bed_ref.py: bed_to_gt).  Code 3 stands for x = the model's moving mean of the site.
"""
from __future__ import annotations

import numpy as np


def mapped_counts(gt, src, flip):
    """gt int8 [nvar, N, 2], src int [K], flip [K] -> uint8 [N, K] with values 0..3, one call at a time."""
    nsamp = gt.shape[1]
    K = len(src)
    out = np.empty((nsamp, K), dtype=np.uint8)
    for k in range(K):
        for i in range(nsamp):
            if src[k] < 0:
                out[i, k] = 3
                continue
            a0, a1 = int(gt[src[k], i, 0]), int(gt[src[k], i, 1])
            if a0 not in (0, 1) or a1 not in (0, 1):
                out[i, k] = 3
            elif flip[k]:
                out[i, k] = (a0 == 0) + (a1 == 0)
            else:
                out[i, k] = a0 + a1
    return out


def first_layer_input(counts, moving_mean):
    """float32 [N, K] the first layer reads: the count, or the site's moving mean where the count is 3."""
    x = np.asarray(counts, dtype=np.float32).copy()
    for i in range(x.shape[0]):
        for k in range(x.shape[1]):
            if counts[i, k] == 3:
                x[i, k] = moving_mean[k]
    return x
