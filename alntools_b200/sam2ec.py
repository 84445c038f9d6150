"""`python -m alntools_b200.sam2ec SAM_FILE|- EC_FILE [-s SAMPLE] [-t TARGETS] [--rangefile F] [-v]`: convert
single-sample SAM text, from a file or from standard input ("-"), into an EC file (sam_utils.convert_sam)."""
import click

from . import utils


@click.command(options_metavar='<options>', context_settings=dict(help_option_names=['-h', '--help']))
@click.argument('sam_file', metavar='sam_file')
@click.argument('ec_file', metavar='ec_file', type=click.Path(resolve_path=True, dir_okay=False, writable=True))
@click.option('-s', '--sample', help="sample identifier (default: the file's base name, 'stdin' for -)")
@click.option('-t', '--targets', metavar='FILE', type=click.Path(exists=True, resolve_path=True, file_okay=True,
                                                                dir_okay=False), help="target file")
@click.option('--rangefile', type=click.Path(exists=False, resolve_path=True, file_okay=True, dir_okay=False,
                                             writable=True), help="range file")
@click.option('-v', '--verbose', count=True, help='enables verbose mode')
def sam2ec(sam_file, ec_file, sample, targets, rangefile, verbose):
    """Convert SAM text (sam_file, or - for standard input) to a binary EC file (ec_file)"""
    from . import sam_utils
    utils.configure_logging(verbose)
    sam_utils.convert_sam(sam_file, ec_file, range_filename=rangefile, sample=sample, target_filename=targets)


if __name__ == "__main__":
    sam2ec()
