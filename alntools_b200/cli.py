"""`python -m alntools_b200 bam2ec|bam2emase ...` with the reference's options (alntools/cli.py:43-89)."""
import click

from . import methods, utils


@click.group(context_settings=dict(help_option_names=['-h', '--help']))
def cli():
    """alntools bam2ec / bam2emase on a B200"""


def _common(fn):
    opts = [
        click.option('-c', '--chunks', default=0, help="number of chunks to process"),
        click.option('-d', '--directory', type=click.Path(exists=True, resolve_path=True, file_okay=False,
                                                          dir_okay=True, writable=True), help="temp directory"),
        click.option('--multisample', is_flag=True),
        click.option('-p', '--number-processes', default=-1, help="number of processes"),
        click.option('--rangefile', type=click.Path(exists=False, resolve_path=True, file_okay=True,
                                                    dir_okay=False, writable=True), help="range file"),
        click.option('-t', '--targets', metavar='FILE', type=click.Path(exists=True, resolve_path=True,
                                                                       file_okay=True, dir_okay=False),
                     help="target file"),
        click.option('-v', '--verbose', count=True, help='enables verbose mode'),
    ]
    for opt in reversed(opts):
        fn = opt(fn)
    return fn


@cli.command('bam2ec', options_metavar='<options>', short_help='convert a BAM file to EC')
@click.argument('bam_file', metavar='bam_file', type=click.Path(exists=True, resolve_path=True, dir_okay=True))
@click.argument('ec_file', metavar='ec_file', type=click.Path(resolve_path=True, dir_okay=False, writable=True))
@click.option('-m', '--mincount', default=1000, help="minimum count")
@click.option('-s', '--sample', help="sample identifier")
@_common
def bam2ec(bam_file, ec_file, chunks, directory, mincount, multisample, number_processes, rangefile, sample,
           targets, verbose):
    """Convert a BAM file (bam_file) to a binary EC file (ec_file)"""
    utils.configure_logging(verbose)
    if multisample:
        if sample:
            print('-s, --sample should NOT be specified with --multisample')
            return
        methods.bam2ec_multisample(bam_file, ec_file, chunks, mincount, directory, number_processes, rangefile,
                                   targets)
    else:
        methods.bam2ec(bam_file, ec_file, chunks, directory, number_processes, rangefile, sample, targets)


@cli.command('bam2emase', options_metavar='<options>', short_help='convert a BAM file to EMASE format')
@click.argument('bam_file', metavar='bam_file', type=click.Path(exists=True, resolve_path=True, dir_okay=True))
@click.argument('emase_file', metavar='emase_file', type=click.Path(resolve_path=True, dir_okay=False,
                                                                    writable=True))
@click.option('-m', '--mincount', default=2000, help="minimum count")
@_common
def bam2emase(bam_file, emase_file, chunks, directory, mincount, multisample, number_processes, rangefile,
              targets, verbose):
    """Convert a BAM file (bam_file) to an EMASE file (emase_file)"""
    utils.configure_logging(verbose)
    if multisample:
        methods.bam2emase_multisample(bam_file, emase_file, chunks, mincount, directory, number_processes,
                                      rangefile, targets)
    else:
        methods.bam2emase(bam_file, emase_file, chunks, directory, number_processes, rangefile, targets)


@cli.command('ec2emase', options_metavar='<options>', short_help='convert a binary EC file to EMASE format')
@click.argument('ec_file', metavar='ec_file', type=click.Path(exists=True, resolve_path=True, dir_okay=False))
@click.argument('emase_file', metavar='emase_file', type=click.Path(resolve_path=True, dir_okay=False))
@click.option('-v', '--verbose', count=True, help='enables verbose mode')
def ec2emase(ec_file, emase_file, verbose):
    """Convert a binary EC format file (ec_file) to EMASE format (emase_file)"""
    utils.configure_logging(verbose)
    methods.ec2emase(ec_file, emase_file)


@cli.command('bam2ec-samples', options_metavar='<options>', short_help='convert several BAM files to one EC file')
@click.argument('ec_file', metavar='ec_file', type=click.Path(resolve_path=True, dir_okay=False, writable=True))
@click.argument('bam_files', metavar='bam_file...', nargs=-1, required=True,
                type=click.Path(exists=True, resolve_path=True, dir_okay=False))
@click.option('-s', '--sample', 'samples', multiple=True, help="sample identifier, once per bam_file, in order")
@click.option('--rangefile', type=click.Path(exists=False, resolve_path=True, file_okay=True, dir_okay=False,
                                             writable=True), help="range file")
@click.option('-t', '--targets', metavar='FILE', type=click.Path(exists=True, resolve_path=True, file_okay=True,
                                                               dir_okay=False), help="target file")
@click.option('-v', '--verbose', count=True, help='enables verbose mode')
def bam2ec_samples(ec_file, bam_files, samples, rangefile, targets, verbose):
    """Convert BAM files (bam_file..., one per sample, read as bam2ec reads one) to one binary EC file (ec_file)
    with one column per sample over one shared EC index"""
    from . import bam_utils
    utils.configure_logging(verbose)
    bam_utils.convert_samples(list(bam_files), ec_file, sample_names=list(samples) or None, target_filename=targets,
                              range_filename=rangefile)


@click.group()
def _merge_commands():
    """commands that work on EC files alone"""


@_merge_commands.command('ec-merge', options_metavar='<options>', short_help='merge EC files into one EC file')
@click.argument('ec_file', metavar='ec_file', type=click.Path(resolve_path=True, dir_okay=False, writable=True))
@click.argument('in_files', metavar='in_ec_file...', nargs=-1, required=True,
                type=click.Path(exists=True, resolve_path=True, dir_okay=False))
@click.option('-s', '--sample', 'samples', multiple=True,
              help="sample identifier, once per column of the inputs, in order")
@click.option('-v', '--verbose', count=True, help='enables verbose mode')
def ec_merge(ec_file, in_files, samples, verbose):
    """Merge binary EC files (in_ec_file..., with one haplotype and target list) into one binary EC file (ec_file)
    with every input's columns over one shared EC index"""
    from . import bin_utils
    utils.configure_logging(verbose)
    bin_utils.merge_ec_files(list(in_files), ec_file, sample_names=list(samples) or None)


# `python -m alntools_b200`: the converter commands of `cli` and the commands on EC files, in one command line.
# `cli` keeps exactly the reference's commands and bam2ec-samples.
main = click.CommandCollection(sources=[cli, _merge_commands], context_settings=dict(help_option_names=['-h', '--help']),
                               help="alntools bam2ec / bam2emase on a B200")
