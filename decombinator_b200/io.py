"""Command line and file output of the decombine path (reference io.py).

Keeps the reference's CLI surface -- ``decombinator {pipeline,decombine,collapse,translate}`` with the
same flags, defaults and destinations (io.py:41-383) --, its programmatic twin ``create_args_dict``
(io.py:391-465) and the exact ``.n12`` text format of ``write_out_intermediate`` (io.py:480-513).
Flags are declared as data so that a flag shared by several stages is only ever added once per parser
(what the reference's handle_clash does, io.py:9-38).
"""
import argparse
import gzip
import os

from . import __version__

# (short, long, kwargs) per stage; order follows the reference's --help
_COMMON = [
    ("-s", "--suppresssummary", dict(action="store_true", help="Suppress the production of summary data log/file")),
    ("-dz", "--dontgzip", dict(action="store_true", help="Stop the output FASTQ files automatically being compressed with gzip")),
    ("-dc", "--dontcount", dict(action="store_true", help="Stop/Block printing the running count")),
    ("-op", "--outpath", dict(type=str, required=False, default="",
                              help="Path to output directory, writes to directory script was called in by default")),
    ("-c", "--chain", dict(type=str, help="TCR chain (a/b/g/d)")),
    ("-pf", "--prefix", dict(type=str, default="dcr_", help='Specify the prefix of the output DCR file. Default = "dcr_"')),
    ("-ds", "--dontsave", dict(action="store_true", help="Don't save output files. For use when writing scripts which use the pipeline.")),
    ("-sa", "--sampling_analysis", dict(action="store_true", help="Saves extra info on R2 V gene and UMI. For use with --writeclusters.")),
]
_DECOMBINE = [
    ("-in", "--infile", dict(type=str, required=True, help="Correctly demultiplexed/processed FASTQ file containing TCR reads")),
    ("-br", "--bc_read", dict(type=str, required=True, help="Which read has bar code (R1,R2). If used, ensure read selected is present in the same directory as the file specified by -in.")),
    ("-dk", "--dontcheck", dict(action="store_true", help="Skip the FASTQ check")),
    ("-ex", "--extension", dict(type=str, default="n12", help='Specify the file extension of the output DCR file. Default = "n12"')),
    ("-or", "--orientation", dict(type=str, default="reverse", help="Specify the orientation to search in (forward/reverse/both). Default = reverse")),
    ("-tg", "--tags", dict(type=str, default="extended", help="Specify which Decombinator tag set to use (extended or original). Default = extended")),
    ("-sp", "--species", dict(type=str, default="human", help="Specify which species TCR repertoire the data consists of (human or mouse). Default = human")),
    ("-N", "--allowNs", dict(action="store_true", help="Whether to allow VJ rearrangements containing ambiguous base calls ('N'). Default = False")),
    ("-ln", "--lenthreshold", dict(type=int, default=130, help="Acceptable threshold for inter-tag (V to J) sequence length. Default = 130")),
    ("-tfdir", "--tagfastadir", dict(type=str, default="Decombinator-Tags-FASTAs", help='Path to folder containing TCR FASTA and Decombinator tag files, for offline analysis. Default = "Decombinator-Tags-FASTAs".')),
    ("-nbc", "--nobarcoding", dict(action="store_true", help="Option to run Decombinator without barcoding, i.e. so as to run on data produced by any protocol.")),
    ("-bl", "--bclength", dict(type=int, default=42, help="Length of barcode sequence, if applicable. Default is set to 42 bp.")),
]
_COLLAPSE = [
    ("-in", "--infile", dict(type=str, required=True, help="File containing raw verbose Decombinator output, i.e. 5 part classifier plus barcode and inter-tag sequence and quality strings")),
    ("-mq", "--minbcQ", dict(type=int, default=20, help="Minimum quality score that barcode nucleotides should be to for that rearrangement to be retained. Default = 20.")),
    ("-bm", "--bcQbelowmin", dict(type=int, default=1, help="Number of nucleotides per barcode whose quality score are allowed to be below -mq and still be retained. Default = 1.")),
    ("-aq", "--avgQthreshold", dict(type=int, default=30, help="Average quality threshold that barcode sequences must remain above for rearrangements to be retained. Default = 30")),
    ("-lv", "--percentlevdist", dict(type=int, default=10, help="Percentage Levenshtein distance that is allowed to estimate whether two sequences within a barcode are derived from the same originator molecule. Default = 10")),
    ("-bc", "--bcthreshold", dict(type=int, default=2, help="Number of sequence edits that are allowed to consider two barcodes to be derived from same originator during clustering. Default = 2.")),
    ("-ex", "--extension", dict(type=str, default="freq", required=False, help="Specify the file extension of the output DCR file. Default = 'freq'")),
    ("-N", "--allowNs", dict(action="store_true", help="Used to allow VJ rearrangements containing ambiguous base calls ('N')")),
    ("-ln", "--lenthreshold", dict(type=int, default=130, required=False, help="Acceptable threshold for inter-tag (V to J) sequence length")),
    ("-di", "--dontcheckinput", dict(action="store_true", help="Override the input file sanity check")),
    ("-bd", "--barcodeduplication", dict(action="store_true", help="Optionally output a file containing the final list of clustered barcodes, and their frequencies")),
    ("-pb", "--positionalbarcodes", dict(action="store_true", help="Instead of inferring random barcode sequences from their context relative to spacer sequences, just take the sequence at the default positions. Useful to salvage runs when R2 quality is terrible.")),
    ("-ol", "--oligo", dict(type=str, required=True, default="m13", help='Choose experimental oligo for correct identification of spacers ["M13", "I8", "I8_single", "NEBIO", "TAKARA"] (default: M13)')),
    ("-wc", "--writeclusters", dict(action="store_true", help="Write cluster data to separate cluster files")),
    ("-uh", "--UMIhistogram", dict(action="store_true", help="Creates histogram of average UMI cluster sizes")),
]
_TRANSLATE = [
    ("-in", "--infile", dict(type=str, required=True, help="File containing 5 part classifier plus barcode and inter-tag sequence and quality strings")),
    ("-sp", "--species", dict(type=str, default="human", required=False, help="Specify which species TCR repertoire the data consists of (human or mouse). Default = human")),
    ("-tg", "--tags", dict(type=str, default="extended", required=False, help="Specify which Decombinator tag set to use (extended or original). Default = extended")),
    ("-npf", "--nonproductivefilter", dict(action="store_true", help="Filter out non-productive reads from the output")),
    ("-tfdir", "--tagfastadir", dict(type=str, default="Decombinator-Tags-FASTAs", required=False, help="Path to folder containing TCR FASTA and Decombinator tag files, for offline analysis. Default = 'Decombinator-Tags-FASTAs'")),
    ("-nbc", "--nobarcoding", dict(action="store_true", help="Option to run CD3translator without barcoding, i.e. so as to run on data produced by any protocol.")),
]

_STAGES = {
    "pipeline": ("Run the entire Decombinator pipeline", (_COMMON, _DECOMBINE, _COLLAPSE, _TRANSLATE)),
    "decombine": ("Decombine TCR reads", (_COMMON, _DECOMBINE)),
    "collapse": ("Collapse barcodes", (_COMMON, _COLLAPSE)),
    "translate": ("Translate Decombinator indexes", (_COMMON, _TRANSLATE)),
}


def _add_flags(parser, groups):
    seen = set()
    for group in groups:
        for short, long_, kw in group:
            if long_ in seen:  # first declaration wins, as with the reference's handle_clash
                continue
            seen.add(long_)
            parser.add_argument(short, long_, **kw)


def create_parser():
    parser = argparse.ArgumentParser(
        description="Decombinator: A fast and efficient tool for the analysis of T-cell receptor repertoire sequences "
                    "produced by deep sequencing. Include a positional argument to run a specific command. "
                    "(B200-native build of the decombine path.)")
    parser.add_argument("-v", "--version", action="version", version=__version__)
    sub = parser.add_subparsers(dest="command", help="Available commands")
    sub.required = False
    for name, (help_, groups) in _STAGES.items():
        _add_flags(sub.add_parser(name, help=help_), groups)
    return parser


def cli_args():
    return vars(create_parser().parse_args())


def create_args_dict(infile: str, chain: str, bc_read: str, suppresssummary: bool = False, dontgzip: bool = False,
                     dontcheck: bool = False, dontcount: bool = False, extension: str = "n12", prefix: str = "dcr_",
                     orientation: str = "reverse", tags: str = "extended", species: str = "human", allowNs: bool = False,
                     lenthreshold: int = 130, tagfastadir: str = "Decombinator-Tags-FASTAs", nobarcoding: bool = False,
                     bclength: int = 42, minbcQ: int = 20, bcQbelowmin: int = 1, avgQthreshold: int = 30,
                     percentlevdist: int = 10, bcthreshold: int = 2, dontcheckinput: bool = False,
                     barcodeduplication: bool = False, positionalbarcodes: bool = False, oligo: str = "M13",
                     writeclusters: bool = False, UMIhistogram: bool = False, nonproductivefilter: bool = False,
                     outpath: str = None, dontsave: bool = False, command: str = None,
                     sampling_analysis: bool = False) -> dict:
    """Argument dictionary for decombinator / collapsinator / cdr3translator (io.py:391-465)."""
    return dict(locals())


def sort_permissions(fl):
    if oct(os.stat(fl).st_mode)[4:] != "666":
        os.chmod(fl, 0o666)


def intermediate_filename(inputargs: dict, suffix: str) -> str:
    """Output name rule of write_out_intermediate (io.py:481-493)."""
    chainnams = {"a": "alpha", "b": "beta", "g": "gamma", "d": "delta"}
    filename_id = os.path.basename(inputargs["infile"]).split(".")[0]
    if inputargs["command"] in ["collapse", "translate"]:
        return inputargs["outpath"] + f"{filename_id}" + suffix
    return inputargs["outpath"] + inputargs["prefix"] + f"{filename_id}" + f"_{chainnams[inputargs['chain'].lower()]}" + suffix


def write_out_intermediate(data: list, inputargs: dict, suffix: str):
    """``.n12`` / ``.freq`` writer: ``", ".join(map(str, row)) + "\\n"`` per row, gzip unless -dz (io.py:480-513)."""
    outfilename = intermediate_filename(inputargs, suffix)
    if hasattr(data, "text"):     # decombine.RowsText: the rows already formatted natively (dcb_format_rows)
        with open(outfilename, "wb") as outfile:
            outfile.write(memoryview(data.text.a) if hasattr(data.text, "a") else data.text)
    else:
        with open(outfilename, "w") as outfile:
            outfile.writelines(", ".join(map(str, line)) + "\n" for line in data)
    if not inputargs["dontgzip"]:
        print("Compressing intermediate output file to", outfilename + ".gz")
        with open(outfilename) as infile, gzip.open(outfilename + ".gz", "wt") as outfile:
            outfile.writelines(infile)
        os.unlink(outfilename)
        outfilename += ".gz"
    sort_permissions(outfilename)


def write_out_translated(data, inputargs: dict):
    """AIRR ``.tsv`` writer: ``DataFrame.to_csv(sep="\\t", index=False)``, gzip unless -dz (io.py:516-548).  `data`: the
    DataFrame of cdr3translator, or the text of translate.translate_tsv (written as it is: the same bytes)."""
    chainnams = {"a": "alpha", "b": "beta", "g": "gamma", "d": "delta"}
    filename_id = os.path.basename(inputargs["infile"]).split(".")[0]
    if inputargs["command"] in ["collapse", "translate"]:
        outfilename = inputargs["outpath"] + f"{filename_id}" + ".tsv"
    else:
        outfilename = inputargs["outpath"] + inputargs["prefix"] + f"{filename_id}" + f"_{chainnams[inputargs['chain'].lower()]}" + ".tsv"
    if hasattr(data, "to_csv"):
        data.to_csv(f"{outfilename}", sep="\t", index=False)
    else:
        with open(outfilename, "wb") as outfile:
            data.write(outfile)
    if not inputargs["dontgzip"]:
        print("Compressing pipeline output file to", outfilename + ".gz")
        with open(outfilename) as infile, gzip.open(outfilename + ".gz", "wt") as outfile:
            outfile.writelines(infile)
        os.unlink(outfilename)
        outfilename += ".gz"
    sort_permissions(outfilename)
