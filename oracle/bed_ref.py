"""Oracle: PLINK 1 .bed records -> the GT cube they stand for (CPU, plain loops).

TEST INFRASTRUCTURE -- see oracle/__init__.py.  Restates the PLINK 1 binary format
(SNP-major, mode byte 0x01) as ``--bed`` reads it, so that the reference's ingest
(oracle/ingest_ref.py: filter_snps, replace_md) can run on a .bed file's content:

  file     = 0x6C 0x1B 0x01, then one record per variant (.bim line)
  record   = ceil(N/4) bytes; sample i is the 2-bit field at bits 2*(i%4) of byte i/4
  field    0 -> (1, 1)   homozygous A1 (A1, .bim column 5, is allele index 1)
           1 -> (-1, -1) missing
           2 -> (0, 1)   heterozygous
           3 -> (0, 0)   homozygous A2
  pad fields of a record's last byte (samples >= N) are not genotypes.
"""
from __future__ import annotations

import numpy as np

CODE_TO_GT = {0: (1, 1), 1: (-1, -1), 2: (0, 1), 3: (0, 0)}


def bed_to_gt(records, nsamp):
    """records: [nvar][ceil(N/4)] bytes (header stripped) -> GT int8 [nvar, N, 2], one call at a time."""
    records = np.asarray(records, dtype=np.uint8)
    nvar = records.shape[0]
    gt = np.empty((nvar, nsamp, 2), dtype=np.int8)
    for v in range(nvar):
        for i in range(nsamp):
            code = (int(records[v, i // 4]) >> (2 * (i % 4))) & 3
            gt[v, i] = CODE_TO_GT[code]
    return gt


def read_bed_file(path, nvar, nsamp):
    """The records of a .bed file after checking its header and size."""
    data = open(path, "rb").read()
    assert data[:3] == b"\x6c\x1b\x01", data[:3]
    rb = (nsamp + 3) // 4
    assert len(data) == 3 + nvar * rb, (len(data), nvar, nsamp)
    return np.frombuffer(data[3:], dtype=np.uint8).reshape(nvar, rb)
