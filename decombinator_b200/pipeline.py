"""Entry point: ``decombinator {decombine|pipeline|collapse|translate}`` (reference pipeline.py:10-53): decombine ->
``.n12`` -> collapse -> ``.freq`` -> translate -> AIRR ``.tsv``, stages chained in memory.

Under ``torchrun`` (WORLD_SIZE > 1) the same commands run one process per GPU: reads are sharded over the ranks for
``decombine``, rows are repartitioned by barcode hash for ``collapse`` (parallel.py); rank 0 writes the files."""
import os
from datetime import datetime

from .decombine import decombinator
from .io import cli_args, write_out_intermediate, write_out_translated


def _world():
    return int(os.environ.get("WORLD_SIZE", "1"))


def run(args=None, cli_args=None):
    """Decombine -> .n12 -> collapse -> .freq -> translate -> .tsv, stages chained in memory (reference pipeline.py:10-38).
    Returns the translated DataFrame (the reference returns nothing; its tests read the files)."""
    return _run(cli_args if cli_args else args, frame=True)


def _run(inputargs, frame):
    """run(); frame=False (the command line): the translate stage hands its .tsv text straight to the writer, and no
    DataFrame is built (nor pandas imported) unless a row needs the host path."""
    start = datetime.now()
    from .collapse import collapsinator
    from .translate import cdr3translator, translate_tsv
    translator = cdr3translator if frame else translate_tsv
    if _world() > 1:
        from . import parallel
        rank, _ = parallel.init_from_env()
        mine, first = parallel.decombinator_shard(inputargs)
        data = parallel.gather_rows(mine)
        if rank == 0 and not inputargs["dontsave"]:
            write_out_intermediate(data, inputargs, ".n12")
        print("Decombinator complete...")
        data = parallel.collapsinator_sharded(inputargs, data=mine, first_index=first)
        if rank == 0 and not inputargs["dontsave"]:
            write_out_intermediate(data, inputargs, ".freq")
        print("Collapsinator complete...")
        if rank != 0:
            return data
        data = translator(data=data, inputargs=inputargs)     # the collapsed rows are few: rank 0 translates them
        print("CDR3translator complete...")
        if not inputargs["dontsave"]:
            write_out_translated(data, inputargs)
        print(f"Pipeline complete in {datetime.now() - start}")
        return data
    inputargs["rows_as_columns"] = True          # the rows stay columnar between the stages (decombine.RowsColumns)
    data = decombinator(inputargs)
    if not inputargs["dontsave"]:
        write_out_intermediate(data, inputargs, ".n12")
    print("Decombinator complete...")
    data = collapsinator(data=data, inputargs=inputargs)
    if not inputargs["dontsave"]:
        write_out_intermediate(data, inputargs, ".freq")
    print("Collapsinator complete...")
    data = translator(data=data, inputargs=inputargs)
    print("CDR3translator complete...")
    if not inputargs["dontsave"]:
        write_out_translated(data, inputargs)
    print(f"Pipeline complete in {datetime.now() - start}")
    return data


def main():
    inputargs = cli_args()
    multi = _world() > 1
    if multi:
        from . import parallel
        rank, _ = parallel.init_from_env()
    else:
        rank = 0
    if inputargs["command"] == "decombine":
        if multi:
            data = parallel.decombinator_sharded(inputargs)
        else:
            inputargs["rows_as_text"] = True      # nothing reads the rows but the .n12 writer
            data = decombinator(inputargs)
        if rank == 0:
            write_out_intermediate(data, inputargs, ".n12")
    elif inputargs["command"] == "collapse":
        from .collapse import collapsinator
        data = parallel.collapsinator_sharded(inputargs) if multi else collapsinator(inputargs=inputargs)
        if rank == 0:
            write_out_intermediate(data, inputargs, ".freq")
    elif inputargs["command"] == "translate":
        from .translate import translate_tsv
        if rank == 0:                                   # the collapsed rows are few: one process translates them
            write_out_translated(translate_tsv(inputargs=inputargs), inputargs)
    else:
        _run(inputargs, frame=False)


if __name__ == "__main__":
    main()
