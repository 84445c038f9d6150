"""One worker of a multi-GPU convert (utils.spawn_ranks): python -m alntools_b200._rank_worker job.json
with RANK / WORLD_SIZE / LOCAL_RANK / MASTER_ADDR / MASTER_PORT in the environment.  The job file names the rank
body: "single" (bam_utils.convert_rank) or "cells" (bam_utils_multisample.convert_files_rank)."""
import json
import os
import sys

from . import bam_utils, bam_utils_multisample, utils

BODIES = {"single": bam_utils.convert_rank, "cells": bam_utils_multisample.convert_files_rank}


def main():
    utils.configure_logging(1 if (os.environ.get("RANK", "0") == "0" and os.environ.get("ALNTOOLS_B200_VERBOSE") == "1") else 0)
    with open(sys.argv[1]) as fh:
        job = json.load(fh)
    summary = BODIES[job["body"]](**job["kwargs"])
    if summary is not None and os.environ.get("ALNTOOLS_B200_SUMMARY"):
        with open(os.environ["ALNTOOLS_B200_SUMMARY"], "w") as fh:
            json.dump(summary, fh)


if __name__ == "__main__":
    main()
