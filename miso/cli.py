"""python -m miso.cli — the reference's command names and options (ref:miso/cli.py:20-253).

infer-object-detector-directory is the runnable command (it needs no CVAT server);
train-object-detector, infer-object-detector and crop-objects talk to a CVAT REST service in the
reference (hard-coded http://cvat:8080) and are outside the accelerated path — they keep their
names and flags and explain that when invoked.
"""
import os
from pathlib import Path

import click

from miso.object_detection.crop import crop_objects as crop_objects_fn
from miso.object_detection.inference import infer_directory as infer_directory_fn


def read_labels(labels_path):
    """labels.txt: one `idx,name` line per class (ref:miso/cli.py:163-168)."""
    labels = []
    with open(labels_path) as fp:
        for line in fp.readlines():
            parts = line.split(",")
            if len(parts) > 1:
                labels.append(parts[1].strip())
    return labels


@click.group()
def cli():
    pass


def _needs_cvat(name):
    raise click.ClickException(
        f"{name} reads its task from a CVAT server (http://cvat:8080) in the reference; the CVAT client is out of "
        "scope of the B200 hot-path build. Use infer-object-detector-directory, or call "
        "miso.object_detection.inference.infer / crop.crop_objects with a Project you built yourself.")


@cli.command()
@click.option('--tasks', type=str, prompt='List of task ids to train on')
@click.option('--model-dir', type=str, default="/obj_det/models", show_default=True)
@click.option('--name', type=str, default="", help='Model name')
@click.option('--batch-size', type=int, default=2)
@click.option('--max-epochs', type=int, default=100)
@click.option('--wsl2', is_flag=True, default=False)
@click.option('--api', type=str, default="v1", show_default=True)
def train_object_detector(tasks, model_dir, name, batch_size, max_epochs, wsl2, api):
    _needs_cvat("train-object-detector")


@cli.command()
@click.option('--tasks', type=str, prompt='List of task ids to infer on')
@click.option('--model-dir', type=str, default="/obj_det/models", show_default=True)
@click.option('--model', type=str, prompt='Name of folder containing model')
@click.option('--threshold', type=float, default=0.5)
@click.option('--batch-size', type=int, default=2)
@click.option("--nv", is_flag=True, default=False)
@click.option("--wsl2", is_flag=True, default=False)
@click.option('--api', type=str, default="v1", show_default=True)
def infer_object_detector(tasks, model_dir, model, threshold, batch_size, nv, wsl2, api):
    _needs_cvat("infer-object-detector")


@cli.command()
@click.option('--tasks', type=str, prompt='List of task ids to crop from')
@click.option('-o', '--output-dir', type=str, default="/obj_det/crops", show_default=True)
@click.option("--wsl2", is_flag=True, default=False)
@click.option('--api', type=str, default="v1", show_default=True)
def crop_objects(tasks, output_dir, wsl2, api):
    _needs_cvat("crop-objects")


@cli.command()
@click.option('-i', '--input-dir', type=str, prompt='Name of folder containing images to infer on')
@click.option('-o', '--output-dir', type=str, prompt='Name of folder to store results')
@click.option('--model-dir', type=str, default="/obj_det/models", show_default=True)
@click.option('--model', type=str, prompt='Name of folder containing model')
@click.option('--threshold', type=float, default=0.5, help='Detection threshold')
@click.option('--batch-size', type=int, default=2)
@click.option('--mask-dir', type=str, default=None,
              help='Also write each crop\'s instance mask (Mask R-CNN models) as a PNG under this folder, same relative path')
def infer_object_detector_directory(input_dir, output_dir, model_dir, model, threshold, batch_size, mask_dir):
    model_path = os.path.join(model_dir, model, "model.pt")
    labels = read_labels(os.path.join(model_dir, model, "labels.txt"))
    if mask_dir is None:
        project = infer_directory_fn(input_dir, model_path, labels, threshold, batch_size)
    else:
        try:
            project = infer_directory_fn(input_dir, model_path, labels, threshold, batch_size, with_masks=True)
        except ValueError as e:
            raise click.ClickException(str(e))
    Path(output_dir).mkdir(parents=True, exist_ok=True)
    crop_objects_fn(project, output_dir, relative_to=input_dir, mask_dir=mask_dir)


if __name__ == "__main__":
    cli()
