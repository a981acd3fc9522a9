"""Place new samples against a sample database: `python -m tracs_b200.query --db db.fasta --msa q1.fasta [q2.fasta ...]`.

The database FASTA is read and ingested on the GPU once (tracs_b200.Database); every --msa file is then swept against it
as the two-file call `python -m tracs_b200.distance --msa q.fasta --msa-db db.fasta` would sweep it, and the output CSV
is byte-identical to what that command writes with the same options (rows are written by the same code).

With --append, each --msa file is placed and then added to the database, so later files are also compared with earlier ones:
the rows of a file are every pair whose later sample is in that file (against the database, the earlier files and the file
itself), as `python -m tracs_b200.distance --msa` on the concatenation of the database and the files lists them."""
import argparse
import sys

from . import api
from .distance import HEADER, read_dates, write_rows


def query(db_file, msa_files, output_file, metadata=None, snp_threshold=2147483647, clock_rate=1e-3 * 29903, trans_rate=73.0,
          trans_threshold=None, precision=0.01, n_cpu=1, append=False):
    dates = read_dates(metadata) if metadata is not None else None
    with api.Database.from_fasta(db_file, n_threads=n_cpu) as db, open(output_file, "w") as out:
        out.write(HEADER)
        for msa in msa_files:
            seqs, names = api.read_fasta(msa, n_cpu)
            if seqs.shape[1] != db.L:
                raise ValueError("%s: sequences of %d sites, the database %s has %d: the alignments must have the same length"
                                 % (msa, seqs.shape[1], db_file, db.L))
            if append:
                r = db.append(seqs, dist=snp_threshold, names=names)
                all_names = db.names
            else:
                r = db.query(seqs, dist=snp_threshold)
                all_names = names + db.names
            write_rows(out, msa, r["rows"].tolist(), r["cols"].tolist(), r["dist"].tolist(), all_names, r["filt"].tolist(),
                       r["ncomp"].tolist(), dates, False, clock_rate, trans_rate, trans_threshold, precision)


def main(argv=None):
    ap = argparse.ArgumentParser(description="SNP and transmission distances of new samples against a sample database (B200); "
                                             "the database is ingested once for all --msa files")
    ap.add_argument("--db", dest="db_file", required=True, help="database alignment, FASTA(.gz)")
    ap.add_argument("--msa", dest="msa_files", required=True, nargs="+", help="query alignments, FASTA(.gz), each as long as the database")
    ap.add_argument("--meta", dest="metadata", default=None)
    ap.add_argument("-o", "--output", dest="output_file", required=True)
    ap.add_argument("-D", "--snp_threshold", type=int, default=2147483647)
    ap.add_argument("--clock_rate", type=float, default=1e-3 * 29903)
    ap.add_argument("--trans_rate", type=float, default=73.0)
    ap.add_argument("-K", "--trans_threshold", type=float, default=None)
    ap.add_argument("--precision", type=float, default=0.01)
    ap.add_argument("-t", "--threads", dest="n_cpu", type=int, default=1)
    ap.add_argument("--append", action="store_true", help="add each --msa file to the database after placing it, so that later "
                                                          "files are also compared with it")
    a = ap.parse_args(argv)
    try:
        query(**vars(a))
    except ValueError as e:
        sys.exit("error: %s" % e)


if __name__ == "__main__":
    main()
