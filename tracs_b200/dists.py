"""All-pairs SNP distance matrix of an alignment, as text (the shape snp-dists / pairsnp users feed to tree building and
hierarchical clustering):

    python -m tracs_b200.dists --msa aln.fasta[.gz] [--msa-db db.fasta[.gz]] -o out.tsv [--csv] [-t THREADS]

Without --msa-db: the square matrix of every sample of --msa against every other (symmetric, zero diagonal). With
--msa-db: the query x db rectangle, rows = the --msa samples, columns = the --msa-db samples (the two-file mode of
pairsnp). Values are the SNP distances of `tracs distance` without -D (tracs_b200.distance_matrix on the GPU); the file
is written by the native writer: a header line (an empty cell, then the column names), then one line per row."""
import argparse

import numpy as np

from . import api


def dists(msa, output, msa_db=None, csv=False, threads=1):
    seqs, names = api.read_fasta(msa, n_threads=threads)
    n_query = None
    col_names = names
    if msa_db is not None:
        db, db_names = api.read_fasta(msa_db, n_threads=threads)
        if len(names) and len(db_names) and seqs.shape[1] != db.shape[1]:
            raise RuntimeError("Error reading FASTA, variable sequence lengths!")
        n_query = len(names)
        col_names = db_names
        seqs = np.concatenate([seqs, db]) if len(db_names) else seqs
    if n_query is not None and (n_query == 0 or len(col_names) == 0):
        m = np.zeros((n_query, len(col_names)), np.int32)  # an empty side: nothing to compute
    else:
        m = api.distance_matrix(seqs, n_query=n_query)
    api.write_distance_matrix(output, m, names, col_names, sep="," if csv else "\t", n_threads=threads)
    return m


def main(argv=None):
    ap = argparse.ArgumentParser(description="All-pairs SNP distance matrix (B200)")
    ap.add_argument("--msa", required=True, help="alignment (FASTA, optionally gzipped)")
    ap.add_argument("--msa-db", dest="msa_db", default=None, help="second alignment: write the --msa x --msa-db rectangle")
    ap.add_argument("-o", "--output", required=True)
    ap.add_argument("--csv", action="store_true", help="comma-separated (default: tab-separated)")
    ap.add_argument("-t", "--threads", type=int, default=1, help="threads for reading the FASTA files and formatting the text")
    a = ap.parse_args(argv)
    dists(a.msa, a.output, msa_db=a.msa_db, csv=a.csv, threads=a.threads)


if __name__ == "__main__":
    main()
