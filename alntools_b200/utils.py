"""Host-side helpers that mirror alntools/utils.py (logging, partition, parse_targets)."""
from collections import OrderedDict
import logging
import os

LOG = None


def get_logger():
    """Same logger name as the reference (utils.py:21-30) so log capture keeps working."""
    global LOG
    if LOG is None:
        LOG = logging.getLogger("alntools.utils")
        LOG.addHandler(logging.NullHandler())
    return LOG


def configure_logging(level):
    """utils.py:33-48: 0 -> WARNING, 1 -> INFO, >=2 -> DEBUG."""
    log = get_logger()
    if not any(isinstance(h, logging.StreamHandler) and not isinstance(h, logging.NullHandler)
               for h in log.handlers):
        handler = logging.StreamHandler()
        handler.setFormatter(logging.Formatter("[alntools] %(message)s"))
        log.addHandler(handler)
    log.setLevel(logging.WARNING if level <= 0 else logging.INFO if level == 1 else logging.DEBUG)


def format_time(start, end):
    """utils.py:51-64."""
    hours, rem = divmod(end - start, 3600)
    minutes, seconds = divmod(rem, 60)
    return "{:0>2}:{:0>2}:{:05.2f}".format(int(hours), int(minutes), seconds)


def delete_file(file_name):
    """Remove a file if it is there (alntools/utils.py: same name, same silence)."""
    try:
        os.remove(file_name)
    except OSError:
        pass


def partition(lst, n):
    """utils.py:67-87: contiguous runs, never an empty trailing partition."""
    q, r = divmod(len(lst), n)
    bounds = [q * i + min(i, r) for i in range(n + 1)]
    parts = []
    for i in range(n):
        piece = lst[bounds[i]:bounds[i + 1]]
        if len(piece) == 0:
            break
        parts.append(piece)
    return parts


def parse_targets(target_file):
    """utils.py:161-178: first whitespace token of every non-'#' line, in file order."""
    targets = OrderedDict()
    with open(target_file, "r") as fh:
        for line in fh:
            if line and line[0] == "#":
                continue
            targets[line.strip().split()[0]] = len(targets)
    return targets


def write_range_file(range_filename, main_targets, haplotypes, references, range_min, range_max):
    """The --rangefile report (alntools/bam_utils.py:735-766, bam_utils_multisample.py:638-668): one line
    per main target, one column per haplotype: max(reference_start) - min(reference_start) + 1 over the
    valid alignments of '<target>_<haplotype>' ('<target>' for the empty haplotype), 0 when that
    reference does not exist or got no valid alignment."""
    tid_of = {}
    for tid, name in enumerate(references):
        tid_of.setdefault(name, tid)                           # gettid: the first reference of that name
    with open(range_filename, "w") as fw:
        fw.write("#\t")
        fw.write("\t".join(haplotypes))
        fw.write("\n")
        for main_target in main_targets:
            vals = []
            for haplotype in haplotypes:
                name = main_target if len(haplotype) == 0 else "{}_{}".format(main_target, haplotype)
                tid = tid_of.get(name, -1)
                if tid < 0 or range_min[tid] > range_max[tid]:
                    vals.append("0")
                else:
                    vals.append(str(int(range_max[tid]) - int(range_min[tid]) + 1))
            fw.write(main_target)
            fw.write("\t")
            fw.write("\t".join(vals))
            fw.write("\n")


def bind_to_gpu_numa_node(device_index):
    """Pin the calling process to the CPUs next to GPU `device_index` (NVML's ideal affinity) BEFORE it allocates
    pinned host buffers: first touch then places them in the GPU's own NUMA node.  With one process per GPU
    and several GPUs copying at once, buffers on the far socket make every host-to-device copy cross the
    socket interconnect.  Returns the CPU list, or None when NVML is not there / has nothing to say."""
    try:
        import pynvml
        pynvml.nvmlInit()
        handle = pynvml.nvmlDeviceGetHandleByIndex(int(device_index))
        n_cpus = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(handle, (n_cpus + 63) // 64)
        cpus = [64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1 and 64 * w + b < n_cpus]
        if not cpus:
            return None
        allowed = os.sched_getaffinity(0)
        cpus = sorted(set(cpus) & allowed) or None
        if cpus:
            os.sched_setaffinity(0, cpus)
        return cpus
    except Exception:
        return None


def requested_gpus(devices):
    """How many GPUs the caller asked for: the `devices` keyword, else the environment variable ALNTOOLS_GPUS
    (the CLI keeps the reference's options, so the environment is its only way to say it), else one."""
    if devices is not None:
        return max(1, int(devices))
    try:
        return max(1, int(os.environ.get("ALNTOOLS_GPUS", "1") or 1))
    except ValueError:
        raise ValueError("ALNTOOLS_GPUS must be a number of GPUs, found %r" % os.environ.get("ALNTOOLS_GPUS"))


def under_launcher():
    """True inside a one-process-per-GPU job (torchrun sets RANK / WORLD_SIZE / LOCAL_RANK)."""
    return int(os.environ.get("WORLD_SIZE", "1") or 1) > 1 and "RANK" in os.environ


def spawn_ranks(n_gpus, kwargs, body="single"):
    """A converter on `n_gpus` GPUs from an ordinary call: one worker process per GPU (the contract of the
    multi-GPU path), each running one rank body (_rank_worker: "single" = bam_utils.convert_rank on its shard of
    the file, "cells" = bam_utils_multisample.convert_files_rank on its run of the files) with `kwargs`; rank 0
    reports the totals."""
    import json
    import socket
    import subprocess
    import sys
    import tempfile
    import time
    with socket.socket() as sock:
        sock.bind(("127.0.0.1", 0))
        port = sock.getsockname()[1]
    with tempfile.TemporaryDirectory(prefix="alntools_b200_") as tmp:
        job = os.path.join(tmp, "job.json")
        with open(job, "w") as fh:
            json.dump({"body": body, "kwargs": kwargs}, fh)
        procs = []
        for rank in range(n_gpus):
            env = dict(os.environ, RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(n_gpus),
                       MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), ALNTOOLS_B200_SUMMARY=os.path.join(tmp, "summary.json"),
                       ALNTOOLS_B200_VERBOSE="1" if get_logger().isEnabledFor(20) else "0")
            procs.append(subprocess.Popen([sys.executable, "-m", "alntools_b200._rank_worker", job], env=env))
        # one worker that fails would leave the others waiting in a collective: when the first non-zero exit code
        # shows up the remaining workers (exactly the processes started above) are terminated
        codes = [None] * n_gpus
        while any(c is None for c in codes):
            for i, p in enumerate(procs):
                if codes[i] is None:
                    codes[i] = p.poll()
            if any(c not in (None, 0) for c in codes):
                for i, p in enumerate(procs):
                    if codes[i] is None:
                        p.terminate()
                for i, p in enumerate(procs):
                    if codes[i] is None:
                        try:
                            codes[i] = p.wait(timeout=20)
                        except subprocess.TimeoutExpired:
                            p.kill()
                            codes[i] = p.wait()
                break
            time.sleep(0.02)
        if any(codes):
            raise RuntimeError("multi-GPU bam2ec failed: worker exit codes %s" % codes)
        with open(os.path.join(tmp, "summary.json")) as fh:
            return json.load(fh)
