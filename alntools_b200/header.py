"""BAM header -> target / haplotype tables (alntools/bam_utils.py:561-633, multisample :399-465).

Stays on the host: O(#@SQ) string work done once per job.  The device only ever sees the resulting
int32 lookups tid -> (main-target index, sorted-haplotype index).
"""
from collections import OrderedDict
import sys

import numpy as np

from . import utils

LOG = utils.get_logger()


class TargetTables(object):
    """main_targets (OrderedDict name -> idx), haplotypes (sorted list), lengths int32[T, H],
    tid_target / tid_hap int32[n_references]."""

    def __init__(self, references, ref_lengths, target_filename=None):
        main_targets = OrderedDict()
        if target_filename:                                   # bam_utils.py:571-579
            main_targets = utils.parse_targets(target_filename)
            if len(main_targets) == 0:
                LOG.error("Unable to parse target file")
                sys.exit(-1)
        refs = list(references)
        cut = [name.rfind("_") for name in refs]              # :584-591: split at the LAST '_' unless it leads
        targets = [name[:i] if i > 0 else name for name, i in zip(refs, cut)]
        haps = [name[i + 1:] if i > 0 else "" for name, i in zip(refs, cut)]
        for target in dict.fromkeys(targets):                 # :596-598: unseen targets in header order
            if target not in main_targets:
                main_targets[target] = len(main_targets)
        self.main_targets = main_targets
        self.haplotypes = sorted(set(haps))                   # :602 ('' sorts first)
        hap_idx = {h: i for i, h in enumerate(self.haplotypes)}
        n = len(refs)
        self.tid_target = np.fromiter(map(main_targets.__getitem__, targets), dtype=np.int32, count=n)
        self.tid_hap = np.fromiter(map(hap_idx.__getitem__, haps), dtype=np.int32, count=n)
        # The reference rebuilds '<target>_<hap>' and looks the name up again (bam_utils.py:800-811);
        # that only differs from the direct tid -> (target, hap) map when two @SQ names collapse to the
        # same pair (e.g. 'a' and 'a_'), which no aligner index produces.  Refuse instead of guessing.
        pair = self.tid_target.astype(np.int64) * len(self.haplotypes) + self.tid_hap
        ordered = np.sort(pair)
        if n > 1 and bool((ordered[1:] == ordered[:-1]).any()):
            seen = {}
            for tid, key in enumerate(pair.tolist()):
                if key in seen:
                    raise ValueError("@SQ names %r and %r map to the same (target, haplotype)"
                                     % (refs[seen[key]], refs[tid]))
                seen[key] = tid
        self.lengths = np.zeros((len(main_targets), len(self.haplotypes)), dtype=np.int32)  # :605
        self.lengths[self.tid_target, self.tid_hap] = np.asarray(ref_lengths, dtype=np.int32)  # :615-633

    def target_section(self):
        """The EC file's targets section as bytes, which only the native tables (bamcols) build: None here, and the
        writer builds it from main_targets and lengths."""
        return None

    @property
    def num_targets(self):
        return len(self.main_targets)

    @property
    def num_haplotypes(self):
        return len(self.haplotypes)
