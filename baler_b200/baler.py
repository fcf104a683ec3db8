"""`baler --project WS PROJ --mode train|compress|decompress` on the B200-native hot path.

Keeps the reference's CLI, per-project config files and output layout (reference baler/baler.py:36-456):
  output/compressed_output/model.pt, compressed.npz {data, names, normalization_features}
    (latent_dtype "q2" ... "q8" adds latent_min, latent_step, latent_block_rows and, below 8 bits, latent_bits:
    baler_b200/latent_q8.py)
  output/decompressed_output/decompressed.npz {data, names}
  output/training/normalization_features.npy, loss_data.npy, activations.npy, model_{epoch}.pt
"""
import os
import time
from math import ceil

import numpy as np

from . import latent_q8
from .modules import helper

__all__ = ("perform_compression", "perform_decompression", "perform_training", "print_info")


def main():
    config, mode, workspace_name, project_name, verbose = helper.get_arguments()
    if os.environ.get("BALER_B200_SEED"):  # reproducible initial weights (the reference seeds only inside train(), after the
        import torch                       # model has been constructed: training.py:168-174)
        torch.manual_seed(int(os.environ["BALER_B200_SEED"]))
    project_path = os.path.join("workspaces", workspace_name, project_name)
    output_path = os.path.join(project_path, "output")
    if mode == "newProject":
        helper.create_new_project(workspace_name, project_name, verbose)
    elif mode == "train":
        perform_training(output_path, config, verbose)
    elif mode == "compress":
        perform_compression(output_path, config, verbose)
    elif mode == "decompress":
        perform_decompression(output_path, config, verbose)
    elif mode == "info":
        print_info(output_path, config)
    elif mode in ("plot", "diagnose", "convert_with_hls4ml"):
        raise NotImplementedError(
            f"mode {mode} is outside the B200 hot path; run the reference tool on the same workspace files")
    else:
        raise NameError("Baler mode " + mode + " not recognised. Use baler --help to see available modes.")


def _latent_size(config, shape, original_shape):
    """reference baler.py:115-141: z = ceil(columns / ratio) (1-D) or ceil(H*W / ratio) (2-D)"""
    if config.data_dimension == 1:
        number_of_columns = shape[1]
        config.latent_space_size = ceil(number_of_columns / config.compression_ratio)
        n_features = number_of_columns
    elif config.data_dimension == 2:
        if config.model_type == "dense":
            number_of_rows, number_of_columns = shape[1], shape[2]
            n_features = number_of_columns * number_of_rows
        else:
            number_of_rows, number_of_columns = original_shape[1], original_shape[2]
            n_features = number_of_columns
        config.latent_space_size = ceil((number_of_rows * number_of_columns) / config.compression_ratio)
    else:
        raise NameError("Data dimension can only be 1 or 2. Got config.data_dimension value = " + str(config.data_dimension))
    config.number_of_columns = number_of_columns
    return n_features, number_of_columns


def perform_training(output_path, config, verbose):
    """reference baler.py:84-207"""
    from . import sharded
    helper.refuse_fp64_training(config)  # precision "fp64": what the float64 trainer does not take, before any work
    sharded.dist_env()  # under torchrun: bind this rank to ITS GPU before helper.process allocates anything on a device
    train_set, test_set, normalization_features, original_shape = helper.process(
        config.input_path, config.custom_norm, config.test_size, config.apply_normalization,
        config.convert_to_blocks if hasattr(config, "convert_to_blocks") else None, verbose,
        precision=getattr(config, "precision", None))
    n_features, number_of_columns = _latent_size(config, train_set.shape, original_shape)
    if verbose:
        print(f"Intitalizing Model with Latent Size - {config.latent_space_size} and Features - {n_features}")
        print(f"Device used for training: {helper.get_device()}")
    model = helper.model_init(config.model_name)(n_features=n_features, z_dim=config.latent_space_size)
    training_path = os.path.join(output_path, "training")
    trained_model = helper.train(model, number_of_columns, train_set, test_set, training_path, config)
    if int(os.environ.get("RANK", "0")) != 0:
        return  # data-parallel launch (torchrun): the replicas are identical, rank 0 writes the files
    if config.apply_normalization:
        np.save(os.path.join(training_path, "normalization_features.npy"), normalization_features)
    if config.separate_model_saving:
        raise NotImplementedError("separate_model_saving needs model.encoder/.decoder, which only PJ_Conv_AE has upstream")
    helper.model_saver(trained_model, os.path.join(output_path, "compressed_output", "model.pt"))
    if verbose:
        print(f"Model saved to {os.path.join(output_path, 'compressed_output', 'model.pt')}")


def perform_compression(output_path, config, verbose):
    """reference baler.py:239-338"""
    print("Compressing...")
    start = time.time()
    normalization_features = []
    if config.apply_normalization:
        normalization_features = np.load(os.path.join(output_path, "training", "normalization_features.npy"))
    compressed, error_bound_batch, error_bound_deltas, error_bound_index = helper.compress(
        model_path=os.path.join(output_path, "compressed_output", "model.pt"), config=config)
    print("Compression took:", f"{(time.time() - start) / 60:.3} minutes")
    if compressed is None:
        return  # sharded launch (torchrun): rank 0 holds the gathered latent and writes the file
    names = np.load(config.input_path)["names"]
    save = np.savez_compressed if config.extra_compression else np.savez
    # latent_dtype "q2" ... "q8": packed codes in `data` plus their per-block parameters (latent_q8.npz_arrays)
    latent = latent_q8.npz_arrays(compressed) if isinstance(compressed, latent_q8.PackedLatent) else {"data": compressed}
    save(os.path.join(output_path, "compressed_output", "compressed.npz"), **latent, names=names,
         normalization_features=normalization_features)
    if getattr(config, "save_error_bounded_deltas", False):
        # reference baler.py:316-338: two gzip'd np.save files of object arrays (per batch: the deltas; the batch indices
        # and the (row-in-batch, column) index arrays)
        import gzip

        def obj(items):
            a = np.empty(len(items), dtype=object)
            for i, it in enumerate(items):
                a[i] = it
            return a

        index = np.empty(2, dtype=object)
        index[0], index[1] = np.asarray(error_bound_batch), obj(error_bound_index)
        for name, arr in (("compressed_deltas.npz.gz", obj([np.asarray(d, dtype=np.float16) for d in error_bound_deltas])),
                          ("compressed_batch_index_metadata.npz.gz", index)):
            with gzip.GzipFile(os.path.join(output_path, "compressed_output", name), "w") as f:
                np.save(file=f, arr=arr, allow_pickle=True)


def perform_decompression(output_path, config, verbose):
    """reference baler.py:341-456: decode, un-normalise with the TRAINING features (fused into the decode
    kernel here), cast columns per `type_list`, write decompressed.npz"""
    print("Decompressing...")
    start = time.time()
    with np.load(config.input_path) as f:
        original_shape = f["data"].shape
    features = None
    if config.apply_normalization:
        print("Un-normalizing...")
        features = np.load(os.path.join(output_path, "training", "normalization_features.npy"))
    blocks = hasattr(config, "convert_to_blocks") and config.convert_to_blocks
    # (kept in the file's dtype: float64 features of a table whose offset dwarfs its spread are applied in float64)
    flat_features = None if features is None else np.asarray(features).reshape(2, -1)
    decompressed, names, _ = helper.decompress(
        model_path=os.path.join(output_path, "compressed_output", "model.pt"),
        input_path=os.path.join(output_path, "compressed_output", "compressed.npz"),
        input_path_deltas=os.path.join(output_path, "compressed_output", "compressed_deltas.npz.gz"),
        input_batch_index=os.path.join(output_path, "compressed_output", "compressed_batch_index_metadata.npz.gz"),
        model_name=config.model_name, config=config, output_path=output_path, original_shape=original_shape,
        renormalize_features=flat_features)
    if decompressed is None:
        return  # sharded launch (torchrun): rank 0 holds the gathered rows and writes the file
    if blocks:
        decompressed = decompressed.reshape(original_shape if config.model_type == "dense"
                                            else (original_shape[0], 1, original_shape[1], original_shape[2]))
    if hasattr(config, "type_list"):
        # reference baler.py:426-435: astype("int") truncates toward zero; result stays in the float array
        for index, t in enumerate(config.type_list):
            if np.dtype(t).kind in "iu":
                decompressed[:, index] = np.trunc(decompressed[:, index])
    print("Decompression took:", f"{(time.time() - start) / 60:.3} minutes")
    save = np.savez_compressed if config.extra_compression else np.savez
    save(os.path.join(output_path, "decompressed_output", "decompressed.npz"), data=decompressed, names=names)


def print_info(output_path, config):
    """reference baler.py:459-508: file-size report"""
    mb = lambda p: os.stat(p).st_size / (1024 * 1024)  # noqa: E731
    original = mb(config.input_path)
    compressed = mb(os.path.join(output_path, "compressed_output", "compressed.npz"))
    decompressed = mb(os.path.join(output_path, "decompressed_output", "decompressed.npz"))
    meta = sum(mb(p) for p in (os.path.join(output_path, "compressed_output", "model.pt"),
                               os.path.join(output_path, "training", "loss_data.npy"),
                               os.path.join(output_path, "training", "normalization_features.npy")))
    print("================================== \n Information about your compression \n================================== ")
    print(f"\nCompressed file is {round(compressed / original, 4) * 100}% the size of the original\n")
    print(f"File size before compression: {round(original, 4)} MB\n")
    print(f"Compressed file size: {round(compressed, 4)} MB\n")
    print(f"De-compressed file size: {round(decompressed, 4)} MB\n")
    print(f"Compression ratio: {round(original / compressed, 4)}\n")
    print(f"The meta-data saved has a total size of: {round(meta, 4)} MB\n")
    print(f"Combined, the actual compression ratio is: {round(original / (compressed + meta), 4)}")
    print("\n ==================================")


if __name__ == "__main__":
    main()
