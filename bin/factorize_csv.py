#!/usr/bin/env python3
"""Train the sparse Poisson factorisation on a CSV-formatted count matrix (B200 path).

Same command line, same output files as the reference driver (bin/factorize_csv.py:20-200 of
mederrata/spmf): `<csv>_<D>D_encoding_lt_<bool>_rn_<bool>.csv` (the encoding matrix, one row per
latent dimension), `..._model_....pkl` (saved state) and `..._representation_....csv` (row index
followed by the row's encoding), written after ADVI calibration.  Differences: the model is
`spmf_b200.PoissonFactorization` (current API of mederrata_spmf/poisson.py instead of the legacy
`PoissonMatrixFactorization` the reference script still imports); the count matrix is held on the
device as CSR; the forest-plot PDF of the reference (matplotlib + arviz, bin/factorize_csv.py:141-183)
is not produced; `--log-transform` is rejected (no CUDA path).  `--checkpoint PATH` writes a training
checkpoint every `--checkpoint-every` epochs and, when PATH exists, resumes the run from it (`-e` counts the
epochs of the whole run); the output files are the same either way.
"""
import argparse
import csv
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def build_parser():
    parser = argparse.ArgumentParser(description='Train PMF on CSV-formatted count matrix')
    parser.add_argument('-f', '--csv-file', nargs='?', type=str, help="Enter the CSV file")
    parser.add_argument('-e', '--epoch', nargs='?', type=int, default=300, help='Enter Epoch value: Default: 300')
    parser.add_argument('-d', '--dimension', nargs='?', type=int, default=2, help='Enter embedding dimension. Default: 2')
    parser.add_argument('-b', '--batch-size', nargs='?', type=int, default=5000, help='Enter batch size. Default: 5000')
    parser.add_argument('-lr', '--learning-rate', nargs='?', type=float, default=0.01, help='Enter float. Default: 0.01')
    parser.add_argument('-c', '--clip-value', nargs='?', type=float, default=3., help='Gradient clip value. Default: 3.0')
    parser.add_argument('-lt', '--log-transform', help='Log-transform?', action='store_true')
    parser.add_argument('-rn', '--row-normalize', help='Row normalize based on counts?', action='store_true')
    parser.add_argument('--sample-size', type=int, default=8, help='Monte-Carlo draws per step (not in the reference CLI)')
    parser.add_argument('--device', type=str, default='cuda', help='CUDA device (not in the reference CLI)')
    parser.add_argument('--checkpoint', type=str, default=None,
                        help='Checkpoint file: written during training; if it exists, training resumes from it '
                             '(-e counts the epochs of the whole run) (not in the reference CLI)')
    parser.add_argument('--checkpoint-every', type=int, default=1,
                        help='Epochs between checkpoints. Default: 1 (not in the reference CLI)')
    return parser


def output_names(csv_file, dimension, log_transform, row_normalize):
    """The three file names of bin/factorize_csv.py:128-131, 136-138, 186-188."""
    tail = f"_lt_{log_transform}_rn_{row_normalize}"
    stem = f"{csv_file}_{dimension}D_"
    return stem + "encoding" + tail + ".csv", stem + "model" + tail + ".pkl", stem + "representation" + tail + ".csv"


def load_counts(path):
    """All rows are data (the reference reads with CsvDataset and no header, bin/factorize_csv.py:75-80)."""
    return np.loadtxt(path, delimiter=",", dtype=np.float32, ndmin=2)


def main(argv=None):
    args = build_parser().parse_args(sys.argv[1:] if argv is None else argv)
    if args.csv_file is None:
        sys.exit("You need to specify a csv file")
    if not os.path.exists(args.csv_file):
        sys.exit("File doesn't exist")

    import torch
    import spmf_b200

    counts = load_counts(args.csv_file)
    N, columns = counts.shape
    dev = torch.device(args.device)
    shard = spmf_b200.CsrShard.from_dense(torch.from_numpy(counts), dev)

    factor = spmf_b200.PoissonFactorization(
        latent_dim=args.dimension, feature_dim=columns, strategy=None, scale_columns=True,
        scale_rows=bool(args.row_normalize), log_transform=bool(args.log_transform),
        u_tau_scale=1.0 / np.sqrt(columns * N), device=dev)      # bin/factorize_csv.py:114-119
    factor.compute_scales(shard)                                 # column scales (:84-96 computes them inline)

    batch = min(args.batch_size, N)
    drop = N >= args.batch_size                                  # drop_remainder=True (:109) when a full batch exists
    factor.calibrate_advi(
        lambda: ({'counts': b} for b in shard.iter_batches(batch, drop_remainder=drop)),
        num_steps=args.epoch, rel_tol=1e-4, clip_value=args.clip_value, learning_rate=args.learning_rate,
        sample_size=args.sample_size,                            # :121-124
        checkpoint_path=args.checkpoint, checkpoint_every=args.checkpoint_every, resume=True)

    enc_name, model_name, rep_name = output_names(args.csv_file, args.dimension, args.log_transform, args.row_normalize)
    print("Saving the encoding matrix")
    with open(enc_name, "w") as f:
        writer = csv.writer(f)
        encoding = factor.encoding_matrix().cpu().numpy().T      # (K, D), one row per latent dimension (:130-134)
        for row in range(encoding.shape[0]):
            writer.writerow(encoding[row, :])

    print("Saving the trained model object")
    factor.save(model_name)

    print("Generating representations")
    with open(rep_name, 'w') as f:
        writer = csv.writer(f)
        for r0 in range(0, N, batch):                            # drop_remainder=False here (:190)
            z = factor.encode(shard.batch(r0, min(batch, N - r0), cache=False)).cpu().numpy()
            for row in range(z.shape[0]):
                writer.writerow(np.concatenate([[r0 + row], z[row, :]]))
    return enc_name, model_name, rep_name


if __name__ == "__main__":
    main()
