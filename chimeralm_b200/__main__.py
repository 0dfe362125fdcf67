"""`chimeralm` command line: `predict`, `filter`, `finetune`, `--version` with the reference's flags
(`chimeralm/__main__.py:248-333`).  Run as `python -m chimeralm_b200 predict in.bam -o out/`.

Differences kept deliberate and small (SURVEY.md N2): the README-documented but unimplemented
options (`-m/--max-sample`, `-l/--limit-batches`, `-p/--progress-bar`, `--random-seed`) are
accepted; the default output directory is resolved BEFORE the writer is built (the reference
raises TypeError when `-o` is omitted); weights come from `--ckpt` or a local path because the
Hub is unreachable offline, and `--seed-weights` selects seeded random-init weights.
"""

from __future__ import annotations

import logging
import os
from collections import Counter
from pathlib import Path

import typer

from . import __version__

log = logging.getLogger("chimeralm")

app = typer.Typer(
    context_settings={"help_option_names": ["-h", "--help"]},
    help="ChimeraLM (B200-native predict path): identify chimera artifacts introduced by whole genome amplification.",
)


def set_logging_level(level: int = logging.INFO) -> None:
    logging.basicConfig(level=level, format="%(message)s")


def version_callback(value: bool):
    if value:
        typer.echo(f"chimeralm-b200 {__version__}")
        raise typer.Exit()


@app.callback()
def main(version: bool = typer.Option(None, "--version", "-V", help="Show the application's version and exit.",
                                      callback=version_callback, is_eager=True)):
    """Main entry point."""


from .predict_worker import predict_rank as _predict_rank  # importable module: mp.spawn pickles the target by name


@app.command()
def predict(
    data_path: Path = typer.Argument(..., help="Path to the dataset"),
    gpus: int = typer.Option(1, "--gpus", "-g", help="Number of GPUs to use"),
    output_path: Path = typer.Option(None, "--output", "-o", help="Output path for predictions"),
    batch_size: int = typer.Option(12, "--batch-size", "-b", help="Batch size"),
    num_workers: int = typer.Option(0, "--workers", "-w", help="BAM ingest threads (0 = all host cores)"),
    ckpt_path: Path = typer.Option(None, "--ckpt", "-c", help="Path to the checkpoint file (.ckpt/.pt/.safetensors)"),
    random: bool = typer.Option(False, "--random", "-r", help="Make the prediction not deterministic"),
    verbose: bool = typer.Option(False, "--verbose", "-v", help="Enable verbose output"),
    max_sample: int = typer.Option(None, "--max-sample", "-m", help="Maximum number of reads to predict"),
    limit_batches: int = typer.Option(None, "--limit-batches", "-l", help="Accepted for README compatibility"),
    progress_bar: bool = typer.Option(False, "--progress-bar", "-p", help="Accepted for README compatibility"),
    random_seed: int = typer.Option(None, "--random-seed", help="Accepted for README compatibility"),
    seed_weights: int = typer.Option(0, "--seed-weights", help="Seed of random-init weights when no --ckpt is given"),
    bucket: bool = typer.Option(False, "--bucket", help="Sort reads by length before batching (less padding)"),
):
    """Predict the given dataset using ChimeraLM."""
    import torch

    set_logging_level(logging.DEBUG if verbose else logging.INFO)
    if not torch.cuda.is_available():
        log.error("No CUDA device: the B200-native predict path has no CPU fallback.")
        raise typer.Exit(2)
    if output_path is None:
        output_path = data_path.with_suffix(".predictions")
    output_path.mkdir(parents=True, exist_ok=True)
    world = max(1, min(gpus, torch.cuda.device_count()))
    if batch_size % world != 0:
        log.error(f"Batch size ({batch_size}) is not divisible by the number of devices ({world}).")
        raise typer.Exit(1)
    if ckpt_path is None:
        log.info(f"No --ckpt: using seeded random-init ChimeraLM weights (seed {seed_weights}); the Hub is unreachable offline")
    args = (world, data_path, output_path, batch_size, ckpt_path, seed_weights, max_sample, bucket, 29500 + os.getpid() % 2000, num_workers)
    if world == 1:
        _predict_rank(0, *args)
    else:
        import torch.multiprocessing as mp

        mp.spawn(_predict_rank, args=args, nprocs=world, join=True)
    log.info(f"Predictions saved to {output_path}")
    log.info(f"Filtering {data_path} by predictions from {output_path}")


def filter_bam_by_predcition(bam_path: Path, prediction_path: Path, *, index: bool = True, output_prediction: bool = False) -> None:
    """`chimeralm/__main__.py:99-153`: drop reads predicted 1, keep reads without a prediction."""
    from .bam import BamReader, BamWriter, coordinate_sorted_header, sorted_records_external
    from .callbacks import load_predictions_from_folder

    predictions = load_predictions_from_folder(prediction_path)
    if not predictions:
        log.warning("No predictions found")
        return
    if output_prediction:
        log.info(f"Writing all predictions to {prediction_path / 'predictions.txt'}")
        with Path(prediction_path / "predictions.txt").open("w") as f:
            for name, label in predictions.items():
                f.write(f"{name}\t{label}\n")
    log.info(f"Loaded {len(predictions)} predictions from {prediction_path}")
    counter = Counter(predictions.values())
    log.info(f"Biological: {counter.get(0, 0)} ({counter.get(0, 0) / len(predictions) * 100:.1f}%), "
             f"Chimera artifact: {counter.get(1, 0)} ({counter.get(1, 0) / len(predictions) * 100:.1f}%)")
    output_path = bam_path.with_suffix(".filtered.bam")
    run_bytes = int(os.environ.get("CLM_SORT_RUN_BYTES", 256 << 20))
    try:
        with BamReader(bam_path) as bam:
            out = BamWriter(output_path, bam.header_bytes())

            def kept():
                for read in bam:
                    # The reference iterates `bam_file.fetch()` (chimeralm/__main__.py:131), which is index-driven and
                    # yields placed reads only: records without a reference (refID -1, the unplaced tail of the file) are
                    # not copied.  A placed read with the unmapped flag (a mate stored at its partner's position) is.
                    if read.ref_id < 0:
                        continue
                    if predictions.get(read.name) == 1:
                        continue
                    out.write(read)
                    yield read

            if index:
                # sorted with bounded memory (runs of CLM_SORT_RUN_BYTES spilled to disk and merged), like `samtools sort`
                sorted_path = output_path.with_suffix(".sorted.bam")
                log.info(f"Sorting {output_path}")
                so = BamWriter(sorted_path, coordinate_sorted_header(bam))
                for r in sorted_records_external(kept(), run_bytes=run_bytes, tmpdir=str(output_path.parent)):
                    so.write(r)
                so.close()
            else:
                for _ in kept():
                    pass
            out.close()
        if index:
            from .bai import index_bam

            log.info(f"Indexing {sorted_path}")
            index_bam(sorted_path)
    except Exception as e:
        log.error(f"Error filtering BAM file: {e}")
        if output_path.exists():
            output_path.unlink()
        raise


@app.command()
def finetune(
    data_path: Path = typer.Argument(..., help="Labelled reads (.fq/.fastq[.gz] or .parquet); ids end in |0 or |1"),
    ckpt_path: Path = typer.Option(None, "--ckpt", "-c", help="Model to start from (.ckpt/.pt/.safetensors)"),
    output_path: Path = typer.Option(..., "--output", "-o", help="Tuned checkpoint (.ckpt, Lightning layout)"),
    epochs: int = typer.Option(3, "--epochs", "-e", help="Passes over the training reads"),
    lr: float = typer.Option(1e-3, "--lr", help="AdamW learning rate"),
    batch_size: int = typer.Option(32, "--batch-size", "-b", help="Reads per batch (batches are bucketed by length)"),
    seed: int = typer.Option(0, "--seed", help="Seed of the batch order and the dropout masks"),
    seed_weights: int = typer.Option(0, "--seed-weights", help="Seed of random-init weights when no --ckpt is given"),
    verbose: bool = typer.Option(False, "--verbose", "-v", help="Enable verbose output"),
):
    """Fine-tune the classification head on labelled reads with the backbone frozen (single GPU)."""
    import torch

    from .train import finetune as run_finetune

    set_logging_level(logging.DEBUG if verbose else logging.INFO)
    if not torch.cuda.is_available():
        log.error("No CUDA device: the B200-native path has no CPU fallback.")
        raise typer.Exit(2)
    if ckpt_path is None:
        log.info(f"No --ckpt: starting from seeded random-init ChimeraLM weights (seed {seed_weights})")
    history = run_finetune(data_path, ckpt_path, output_path, epochs=epochs, lr=lr, batch_size=batch_size, seed=seed,
                           seed_weights=seed_weights)
    log.info(f"mean loss per epoch: {', '.join(f'{h:.4f}' for h in history)}")
    log.info(f"Tuned checkpoint saved to {output_path}")


@app.command()
def filter(  # noqa: A001 - reference command name
    bam_path: Path = typer.Argument(..., help="Path to the BAM file"),
    predictions_path: Path = typer.Argument(..., help="Path to the predictions file"),
    output_prediction: bool = typer.Option(False, "--output-prediction", "-p", help="write summary of the predictions"),
    verbose: bool = typer.Option(False, "--verbose", "-v", help="Enable verbose output"),
):
    """Filter the BAM file by predictions."""
    set_logging_level(logging.DEBUG if verbose else logging.INFO)
    log.info(f"Filtering {bam_path} by predictions from {predictions_path}")
    filter_bam_by_predcition(bam_path, predictions_path, index=True, output_prediction=output_prediction)


if __name__ == "__main__":
    app()
