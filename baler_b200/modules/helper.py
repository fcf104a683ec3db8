"""Orchestration helpers with the reference's signatures (reference baler/modules/helper.py): what
`baler.py` calls for `--mode train|compress|decompress`.  Data loading and file layout are host
Python; every numeric step goes to libbaler_b200 (CUDA)."""
import argparse
import importlib
import os
import sys
from math import ceil

import numpy as np
import torch

from .. import engine, latent_q8
from . import data_processing, models, training

sys.path.append(os.getcwd())


class Config:
    """Namespace the per-project `set_config(c)` fills (reference helper.py:150-179: a dataclass used as a
    class-level namespace; attributes that are never set raise AttributeError when read).
    Extra, optional knobs of this implementation (absent = reference behaviour):
      precision        "auto" | "fp32" | "split16" | "fast" | "fp64"   arithmetic of the fused encode/decode kernels;
                       "fp64" computes in float64 like the reference's float64 models (its files to ~1e-15, integer
                       columns equal): dense models of <= 256 columns (AE, AE_Dropout_BN, CFD_dense_AE), float64 files
                       normalised in float64 on the device, float32 files in float32 as numpy does; not with
                       save_error_bounded_deltas.  "fp64" also governs --mode train: the float64 training step
                       (float64 parameters, gradients and Adam state; the reference's training to ~1e-14) for AE and
                       CFD_dense_AE of <= 100 columns with the MSE loss or l1_in_training, float64 files normalised in
                       float64 on the device; AE_Dropout_BN with dropout_stream = "torch" (below); Conv_AE and
                       loss_function_swae are refused.  The other values leave training on its default step (split16
                       tensor cores, fp32 for the L1 chain)
      dropout_stream   "torch": AE_Dropout_BN under precision "fp64" draws its dropout masks on the device from torch's
                       default CPU generator, exactly the masks the reference's run draws, and leaves the generator where
                       the reference's would be: the float64 run then reproduces the reference's training.  One process,
                       batch_size <= 4 rows x the GPU's SMs (592 on a B200).  Without it AE_Dropout_BN is not trained
                       in float64 (a float64 run with other masks is no closer to the reference than split16); with any
                       other precision the key is refused
      latent_dtype     "float64" (AE default, what the reference writes; any model under "fp64") | "float32" | "float16"
                       | "q8": uint8 codes with a float32 (min, step) per latent column and 128-row block (latent_q8),
                       z + 8 z / 128 bytes per row (15.9 for z = 15, against 120 as float64 and 30 as float16); every
                       latent value within half its block's step
                       | "q2" ... "q7": the same with b-bit codes, 2^b - 2 steps per block column, packed row by row:
                       ceil(z b / 8) + 8 z / 128 bytes per row (8.94 for z = 15 at "q4"), the step / 2 error growing by
                       about 2x per bit removed.  decompress recognises a quantised file by itself.  Not with precision
                       "fp64"; another "q..." value is refused
      l1_in_training   bool: add reg_param * L1 chain to the training loss (dead code upstream, SURVEY F2)
    No key is needed for tables larger than device memory: --mode train normalises the table in row chunks, keeps it
    resident when it fits the device memory the trainer leaves (training.device_table_budget), and otherwise streams
    every epoch and validation from host memory through two device windows of whole batches, with the same results.
    """

    model_type = str  # reference helper.py:163: defaults to the *type* `str`


def get_arguments():
    """`baler --project WORKSPACE PROJECT --mode MODE [--verbose]` (reference helper.py:34-101)"""
    parser = argparse.ArgumentParser(
        prog="baler",
        description="Baler (B200-native hot path): train / compress / decompress with fused CUDA autoencoder kernels.",
        formatter_class=argparse.RawTextHelpFormatter,
    )
    parser.add_argument("--mode", type=str, required=True, help="newProject, train, compress, decompress, info")
    parser.add_argument("--project", type=str, required=True, nargs=2, metavar=("WORKSPACE", "PROJECT"),
                        help="workspace and project, e.g. --project CMS_workspace CMS_project_v1")
    parser.add_argument("--verbose", dest="verbose", action="store_true", help="Verbose mode")
    parser.set_defaults(verbose=False)
    args = parser.parse_args()
    workspace_name, project_name = args.project
    if args.mode == "newProject":
        config = None
    else:
        config = Config
        importlib.import_module(
            f"workspaces.{workspace_name}.{project_name}.config.{project_name}_config").set_config(config)
    return config, args.mode, workspace_name, project_name, args.verbose


def create_new_project(workspace_name, project_name, verbose=False, base_path="workspaces"):
    """reference helper.py:104-147: directory skeleton + default config"""
    workspace_path = os.path.join(base_path, workspace_name)
    project_path = os.path.join(workspace_path, project_name)
    if os.path.exists(project_path):
        print(f"The workspace and project ({project_path}) already exists.")
        return
    os.makedirs(project_path)
    for d in (os.path.join(workspace_path, "data"), os.path.join(project_path, "config"),
              os.path.join(project_path, "output", "compressed_output"),
              os.path.join(project_path, "output", "decompressed_output"),
              os.path.join(project_path, "output", "plotting"), os.path.join(project_path, "output", "training")):
        if verbose:
            print(f"Creating directory {d}...")
        os.makedirs(d, exist_ok=True)
    with open(os.path.join(project_path, "config", f"{project_name}_config.py"), "w") as f:
        f.write(create_default_config(workspace_name, project_name))


_DEFAULTS = [  # same keys and values as the reference's template (helper.py:182-232)
    ("input_path", None), ("data_dimension", 1), ("compression_ratio", 2.0), ("apply_normalization", True),
    ("model_name", "AE"), ("model_type", "dense"), ("epochs", 5), ("lr", 0.001), ("batch_size", 512),
    ("early_stopping", True), ("lr_scheduler", True), ("early_stopping_patience", 100), ("min_delta", 0),
    ("lr_scheduler_patience", 50), ("custom_norm", False), ("reg_param", 0.001), ("RHO", 0.05), ("test_size", 0),
    ("extra_compression", False), ("intermittent_model_saving", False), ("intermittent_saving_patience", 100),
    ("mse_avg", False), ("mse_sum", True), ("emd", False), ("l1", True), ("activation_extraction", False),
    ("deterministic_algorithm", True), ("separate_model_saving", False), ("save_error_bounded_deltas", False),
]


def create_default_config(workspace_name, project_name):
    lines = ["", "# === Configuration options ===", "", "def set_config(c):"]
    for key, val in _DEFAULTS:
        if key == "input_path":
            val = f"workspaces/{workspace_name}/data/{project_name}_data.npz"
        lines.append(f"    c.{key:<29}= {val!r}")
    return "\n".join(lines) + "\n"


def model_init(model_name):
    return data_processing.initialise_model(model_name)


def numpy_to_tensor(data):
    return torch.from_numpy(data)


def normalize(data, custom_norm):
    """reference helper.py:261-274 (per column / per pixel over axis 0)"""
    return data_processing.normalize(data, custom_norm)


def renormalize(data, true_min_list, feature_range_list):
    """reference helper.py:322-333"""
    return data_processing.renormalize_func(data, true_min_list, feature_range_list)


def process(input_path, custom_norm, test_size, apply_normalization, convert_to_blocks, verbose, precision=None):
    """reference helper.py:277-319 -> (train_set, test_set, normalization_features, original_shape).
    `precision` (optional, not in the reference signature): "fp64" normalises a float64 file in float64 on the device,
    bit-equal to the reference's numpy (float32 files stay float32-normalised, as upstream)."""
    data = np.load(input_path)["data"]
    if verbose:
        print("Original Dataset Shape - ", data.shape)
    original_shape = data.shape
    if convert_to_blocks:
        data = data_processing.convert_to_blocks_util(convert_to_blocks, data)
    if training.is_fp64(precision):
        engine.require_cuda()  # the float64 trainer, like every compute path, has no CPU fallback
    if training.is_fp64(precision) and data.dtype == np.float64 and data.size:
        if apply_normalization:
            print("Normalizing the data...")
        normalization_features, data = data_processing.minmax_normalize_f64(data, apply_normalization and not custom_norm)
    else:
        normalization_features = data_processing.find_minmax(data)
        if apply_normalization:
            print("Normalizing the data...")
            data = normalize(data, custom_norm)
    if not test_size:
        train_set = test_set = data
    else:
        from sklearn.model_selection import train_test_split

        train_set, test_set = train_test_split(data, test_size=test_size, random_state=1)
    return train_set, test_set, normalization_features, original_shape


def _npz_shape(path, key="data"):
    """shape of array `key` of an .npz file from its header, without reading the array"""
    import zipfile
    with zipfile.ZipFile(path) as z, z.open(key + ".npy") as f:
        version = np.lib.format.read_magic(f)
        read = np.lib.format.read_array_header_1_0 if version == (1, 0) else np.lib.format.read_array_header_2_0
        return read(f)[0]


def refuse_fp64_training(config):
    """--mode train with config.precision == "fp64": NotImplementedError naming what the float64 trainer does not take,
    before any file is read or written (training.refuse_fp64_training).  True when "fp64" trains.  Other precisions:
    the dropout_stream key and AE_Dropout_BN's per-rank batch under torchrun (training.refuse_dbn_rank_share)."""
    stream = getattr(config, "dropout_stream", None)
    if not training.is_fp64(getattr(config, "precision", None)):
        training.refuse_dropout_stream(config.model_name, getattr(config, "precision", None), stream)
        training.refuse_dbn_rank_share(config.model_name, config.batch_size, int(os.environ.get("WORLD_SIZE", "1")))
        return False
    blocks = getattr(config, "convert_to_blocks", None)
    shape = _npz_shape(config.input_path)
    n_features = int(blocks[1]) * int(blocks[2]) if blocks else int(np.prod(shape[1:]))
    training.refuse_fp64_training(config.model_name, n_features,
                                  getattr(config, "custom_loss_function", None) == "loss_function_swae",
                                  dropout_stream=stream, batch_size=config.batch_size,
                                  world=int(os.environ.get("WORLD_SIZE", "1")))
    return True


def train(model, number_of_columns, train_set, test_set, project_path, config):
    return training.train(model, number_of_columns, train_set, test_set, project_path, config)


def model_saver(model, model_path):
    return data_processing.save_model(model, model_path)


def detacher(tensor):
    return tensor.cpu().detach().numpy()


def get_device():
    """reference helper.py:425-439 - here a CUDA device is mandatory"""
    engine.require_cuda()
    return torch.device("cuda:0")


def _latent_np_dtype(model, config):
    """numpy type of the latent compress writes, or the latent_dtype name ("q2" ... "q8") of a quantised latent"""
    name = getattr(config, "latent_dtype", None)
    if name is None:
        return np.float64 if model.dtype == torch.float64 or _fp64(config) else np.float32
    if latent_q8.bits_of(name) is not None:
        return name
    return np.dtype(name).type


def _fp64(config):
    """config.precision == "fp64": the float64 chain; refuses what it does not do before anything is read or written"""
    bits = latent_q8.bits_of(getattr(config, "latent_dtype", None))  # (ValueError for an unknown "q..." value)
    if engine.PRECISIONS.get(getattr(config, "precision", "auto")) != engine.BB_PREC_FP64:
        return False
    if bits is not None:
        raise NotImplementedError("precision='fp64' does not write or read a quantised latent (latent_dtype='q%d'): the "
                                  "%d-bit codes discard far more than float64 arithmetic gains; use another precision or "
                                  "latent_dtype" % (bits, bits))
    if getattr(config, "save_error_bounded_deltas", False):
        raise NotImplementedError("precision='fp64' does not compute error-bounded deltas (save_error_bounded_deltas); "
                                  "use another precision for them")
    return True


def _refuse_fp64_shape(model):
    """NotImplementedError naming the chain when the float64 kernel does not take `model` (Conv_AE, widths > 256)"""
    if isinstance(model, models.Conv_AE):
        raise NotImplementedError("precision='fp64' takes dense chains only; Conv_AE unrolls to dense layers up to %d wide"
                                  % model.q_z_mid_dim)
    dims = [model.n_features, *model.hidden, model.z_dim]
    msg = engine.fp64_refusal({"encoder": dims, "decoder": dims[::-1]})
    if msg:
        raise NotImplementedError(msg)


def compress(model_path, config):
    """reference helper.py:473-616 -> (compressed ndarray, eb_batch, eb_deltas, eb_index).
    Normalisation uses THIS file's column min/max (helper.py:500-502), fused into the encode kernel."""
    from .. import sharded
    fp64 = _fp64(config)
    rank, world = sharded.dist_env()  # under torchrun: this rank's GPU, before anything touches a device
    loaded = np.load(config.input_path)
    data_before = loaded["data"]
    original_shape = data_before.shape
    if hasattr(config, "convert_to_blocks") and config.convert_to_blocks:
        data_before = data_processing.convert_to_blocks_util(config.convert_to_blocks, data_before)
    conv = False
    if config.data_dimension == 1:
        number_of_columns = len(loaded["names"])
        config.latent_space_size = ceil(number_of_columns / config.compression_ratio)
        config.number_of_columns = number_of_columns
        n_features = number_of_columns
    elif config.data_dimension == 2:
        if config.model_type == "dense":
            number_of_rows, config.number_of_columns = data_before.shape[1], data_before.shape[2]
            n_features = number_of_rows * config.number_of_columns
        else:  # convolutional (reference helper.py:521-524): sizes come from the ORIGINAL snapshot shape
            conv = True
            number_of_rows, config.number_of_columns = original_shape[1], original_shape[2]
            n_features = config.number_of_columns
        config.latent_space_size = ceil((number_of_rows * config.number_of_columns) / config.compression_ratio)
    else:
        raise NameError("Data dimension can only be 1 or 2. Got config.data_dimension = " + str(config.data_dimension))
    model = data_processing.load_model(data_processing.initialise_model(config.model_name), model_path,
                                       n_features=n_features, z_dim=config.latent_space_size)
    model.eval()
    if fp64:
        _refuse_fp64_shape(model)
    normalise = bool(config.apply_normalization) and not config.custom_norm
    if config.apply_normalization:
        print("Normalizing...")
    table = None
    if fp64 and data_before.dtype != np.float32:
        # the float64 chain normalises a float64 table in float64 on the device (bb_compress_host_f64)
        table = engine.host_convert(data_before.reshape(data_before.shape[0], -1), np.float64)
    elif normalise and data_before.dtype == np.float64 and data_before.size:
        # a float64 file whose offset dwarfs its spread is normalised here in float64, as the reference's numpy does
        # (data_processing.F32_OFFSET_LIMIT); the kernels then take the normalised float32 table as it is
        flat64 = data_before.reshape(data_before.shape[0], -1)
        shard_stats = None
        if world > 1:  # every rank holds the file: same decision everywhere, statistics from the row shards
            lo64, hi64 = sharded.row_range(len(flat64), rank, world)

            def shard_stats(_flat):
                f = sharded.global_minmax(_flat[lo64:hi64])
                return f[0], f[0] + f[1]
        st = data_processing.float64_stats(flat64, shard_stats)
        if st is not None:
            table = np.ascontiguousarray(data_processing.normalize_float64_host(flat64, st[0], st[1], np.float32))
            normalise = False
    if table is None:
        table = engine.host_convert(data_before.reshape(data_before.shape[0], -1), np.float32)
    codec = model.codec(data_before.shape[1], data_before.shape[2]) if conv else model.codec()
    if getattr(config, "save_error_bounded_deltas", False):
        return _compress_with_deltas(codec, model, table, normalise, config, rank, world)
    bits = latent_q8.bits_of(getattr(config, "latent_dtype", None))
    if bits is not None:
        return _compress_packed(codec, table, normalise, config, rank, world, bits), [], [], []
    if world == 1:
        compressed, _ = codec.compress_host(table, recompute_minmax=normalise,
                                            z_dtype=_latent_np_dtype(model, config),
                                            precision=getattr(config, "precision", "auto"))
        return compressed, [], [], []
    # launched under torchrun: rows are sharded contiguously over the ranks; the only exchange on the way in is the
    # 2 x C column min / max of the whole file, rank 0 collects the latent rows (the other ranks return None)
    lo, hi = sharded.row_range(len(table), rank, world)
    shard = table[lo:hi]
    feats = sharded.global_minmax(shard) if normalise else None
    if len(shard):
        z, _ = codec.compress_host(shard, features=feats, z_dtype=_latent_np_dtype(model, config),
                                   precision=getattr(config, "precision", "auto"))
    else:
        z = np.empty((0, config.latent_space_size), dtype=_latent_np_dtype(model, config))
    return sharded.gather_rows_to_rank0(z, len(table)), [], [], []


def _compress_packed(codec, table, normalise, config, rank, world, bits):
    """latent_dtype "q2" ... "q8": the quantised latent (latent_q8.PackedLatent of numpy arrays).  Under torchrun the shards
    start on the 128-row blocks of the file, so each rank's blocks are the file's and rank 0's gathered result is the
    one-process file byte for byte; the other ranks return None."""
    from .. import sharded
    precision = getattr(config, "precision", "auto")
    if world == 1:
        return codec.compress_host_packed(table, bits, recompute_minmax=normalise, precision=precision)[0]
    n = len(table)
    lo, hi = sharded.row_range(n, rank, world, latent_q8.BLOCK_ROWS)
    shard = table[lo:hi]
    feats = sharded.global_minmax(shard) if normalise else None
    q = (codec.compress_host_packed(shard, bits, features=feats, precision=precision)[0] if len(shard)
         else latent_q8.empty_packed(0, codec.z_dim, bits))
    return _gather_packed(q, n)


def _gather_packed(q, n_rows):
    """this rank's block-aligned share of a quantised latent -> the whole PackedLatent on rank 0 (codes by rows,
    parameters by blocks: the block ranges of aligned row shards are row_range of the block count), None on the others"""
    from .. import sharded
    codes = sharded.gather_rows_to_rank0(q.codes, n_rows, align=latent_q8.BLOCK_ROWS)
    mins = sharded.gather_rows_to_rank0(q.lo, latent_q8.n_blocks(n_rows))
    steps = sharded.gather_rows_to_rank0(q.step, latent_q8.n_blocks(n_rows))
    return None if codes is None else latent_q8.PackedLatent(codes, mins, steps, q.bits)


def _compress_with_deltas(codec, model, table, normalise, config, rank=0, world=1):
    """reference helper.py:583-611 with config.save_error_bounded_deltas: every batch is encoded, decoded again and
    compared with its (normalised) input; elements whose relative error exceeds config.error_bounded_requirement percent
    get a float16 delta (helper.save_error_bounded_requirement, helper.py:442-470).  Here the table goes through the GPU in
    row chunks: encode, decode, one scan kernel (bb_error_bounded_deltas_f32); the hits are regrouped per batch of
    config.batch_size rows on the host, in the reference's (batch index, deltas, (row-in-batch, column)) lists.
    Launched under torchrun every rank scans its contiguous row range (hits carry GLOBAL row numbers), rank 0 collects the
    latent rows and the hit lists and regroups them; the other ranks return (None, [], [], []).
    latent_dtype "q2" ... "q8": each chunk's latent is quantised, and the deltas correct
    decode(dequantise(quantise(encode(x)))), the rows decompress reproduces; shards and chunks start on 128-row blocks."""
    from .. import engine, sharded
    n, bs = len(table), int(config.batch_size)
    z_dtype = _latent_np_dtype(model, config)
    bits = latent_q8.bits_of(z_dtype)
    lo, hi = sharded.row_range(n, rank, world, latent_q8.BLOCK_ROWS if bits else 1)
    shard = table[lo:hi]
    compressed = (latent_q8.empty_packed(hi - lo, codec.z_dim, bits) if bits
                  else np.empty((hi - lo, codec.z_dim), dtype=z_dtype))
    mn = rg = None
    if normalise and n:
        # this file's own [min; range] (helper.py:500-502), over all ranks' rows
        feats = data_processing.find_minmax(table) if world == 1 else sharded.global_minmax(shard)
        mn, rg = torch.from_numpy(np.ascontiguousarray(feats[0])).cuda(), torch.from_numpy(np.ascontiguousarray(feats[1])).cuda()
    rows, cols, deltas = [], [], []
    chunk = 1 << 20
    for r0 in range(0, hi - lo, chunk):
        x = torch.from_numpy(shard[r0:r0 + chunk]).cuda()
        z = codec.encode(x, mn, rg, precision=getattr(config, "precision", "auto"))
        if bits:  # (chunk is a multiple of the block)
            qz = codec.quantize_packed(z, bits)
            b0 = r0 // latent_q8.BLOCK_ROWS
            compressed.codes[r0:r0 + chunk] = qz.codes.cpu().numpy()
            compressed.lo[b0:b0 + len(qz.lo)] = qz.lo.cpu().numpy()
            compressed.step[b0:b0 + len(qz.step)] = qz.step.cpu().numpy()
            z = codec.dequantize_packed(qz)
        else:
            compressed[r0:r0 + chunk] = z.cpu().numpy().astype(z_dtype, copy=False)
        y = codec.decode(z, precision=getattr(config, "precision", "auto"))  # still normalised, as upstream compares it
        r, c, d = engine.error_bounded_deltas(x, y, mn, rg, config.error_bounded_requirement, row0=lo + r0)
        rows.append(r); cols.append(c); deltas.append(d)
    rows = np.concatenate(rows) if rows else np.empty(0, np.int64)
    cols = np.concatenate(cols) if cols else np.empty(0, np.int64)
    deltas = np.concatenate(deltas) if deltas else np.empty(0, np.float16)
    if world > 1:
        compressed = _gather_packed(compressed, n) if bits else sharded.gather_rows_to_rank0(compressed, n)
        hits = sharded.gather_objects_to_rank0((rows, cols, deltas))
        if rank != 0:
            return None, [], [], []
        rows, cols, deltas = (np.concatenate([h[i] for h in hits]) for i in range(3))  # rank order = row order
    print("Total Deltas Found - ", len(rows))
    # upstream appends an entry for EVERY batch (its `len(index) > 0` test is on a 2-tuple); batches without a hit get
    # empty lists here (upstream would reuse the previous batch's deltas or crash on the first one)
    batch_of = rows // bs
    cuts = np.searchsorted(batch_of, np.arange((n + bs - 1) // bs + 1))
    eb_batch, eb_deltas, eb_index = [], [], []
    for b in range(len(cuts) - 1):
        lo, hi = cuts[b], cuts[b + 1]
        eb_batch.append(b)
        eb_deltas.append(list(deltas[lo:hi]))
        eb_index.append((rows[lo:hi] - b * bs, cols[lo:hi]))
    return compressed, eb_batch, eb_deltas, eb_index


def _apply_deltas(decompressed, input_path_deltas, input_batch_index, batch_size, col_scale):
    """reference helper.py:655-665, 708-718: out[row][col] -= delta for every stored delta; `col_scale` = the range of each
    column when un-normalisation is fused into the decode kernel ((y - d) * range + min == y * range + min - d * range)"""
    import gzip
    loaded_deltas = np.load(gzip.GzipFile(input_path_deltas, "r"), allow_pickle=True)
    loaded_index = np.load(gzip.GzipFile(input_batch_index, "r"), allow_pickle=True)
    batches, index = loaded_index[0], loaded_index[1]
    added = 0
    for i, b in enumerate(batches):
        d = np.asarray(loaded_deltas[i], dtype=np.float64)
        r, c = np.asarray(index[i][0], dtype=np.int64), np.asarray(index[i][1], dtype=np.int64)
        if len(d) == 0:
            continue
        step = d if col_scale is None else d * np.asarray(col_scale, dtype=np.float64)[c]
        np.subtract.at(decompressed, (int(b) * batch_size + r, c), step.astype(decompressed.dtype))
        added += len(d)
    print("Total Deltas Added - ", added)
    return decompressed


def decompress(model_path, input_path, input_path_deltas, input_batch_index, model_name, config, output_path,
               original_shape, renormalize_features=None):
    """reference helper.py:619-733 -> (decompressed ndarray, names, normalization_features).
    `renormalize_features` ([min; range], optional, not in the reference signature) fuses the
    un-normalisation of baler.py:410-424 into the decode kernel."""
    from .. import sharded
    fp64 = _fp64(config)
    rank, world = sharded.dist_env()  # under torchrun: this rank's GPU, before anything touches a device
    loaded = np.load(input_path)
    quant = latent_q8.read(loaded) if latent_q8.in_file(loaded) else None  # (checks the arrays before any work)
    if quant is not None and fp64:
        raise NotImplementedError("%s holds a %d-bit latent (latent_dtype='q%d'), which precision='fp64' does not read"
                                  % (input_path, quant.bits, quant.bits))
    data, names, normalization_features = loaded["data"], loaded["names"], loaded["normalization_features"]
    latent_space_size = data.shape[1] if quant is None else quant.lo.shape[1]  # (packed rows are narrower than the latent)
    model_dict = torch.load(str(model_path), map_location="cpu")
    # the reference reads len() of the last state-dict entry, which crashes on AE_Dropout_BN's
    # num_batches_tracked scalar (SURVEY F7a); take the last tensor that has a length instead
    number_of_columns = [len(v) for v in model_dict.values() if getattr(v, "ndim", 0) >= 1][-1]
    model = data_processing.load_model(data_processing.initialise_model(config.model_name), model_path,
                                       n_features=number_of_columns, z_dim=latent_space_size)
    model.eval()
    if fp64:
        _refuse_fp64_shape(model)
        data = engine.host_convert(data, np.float64)  # the latent goes to the float64 chain as float64
    if quant is None and data.dtype not in (np.float16, np.float32, np.float64):
        data = data.astype(np.float32)
    out_dtype = np.float64 if model.dtype == torch.float64 else np.float32
    conv = config.data_dimension == 2 and config.model_type == "convolutional"
    if conv:  # block shape: convert_to_blocks = [1, h, w], else the whole snapshot
        blocks = getattr(config, "convert_to_blocks", None)
        h, w = (int(blocks[1]), int(blocks[2])) if blocks else (original_shape[1], original_shape[2])
        codec = model.codec(h, w)
    else:
        codec = model.codec()
    host_renorm = None
    if renormalize_features is not None and out_dtype == np.float64 and not fp64:
        f64 = np.asarray(renormalize_features, dtype=np.float64).reshape(2, -1)
        if data_processing._ill_conditioned(f64[0], f64[0] + f64[1]):
            # float32 could not hold y * range + min (data_processing.F32_OFFSET_LIMIT): decode to normalised values and
            # un-normalise in float64 on the host, as the reference's renormalize_func does
            host_renorm, renormalize_features = f64, None
    precision = getattr(config, "precision", "auto")

    def run(lo, hi):  # rows [lo, hi) of the file
        if quant is not None:
            return codec.decompress_host_packed(latent_q8.rows(quant, lo, hi), features=renormalize_features,
                                                y_dtype=out_dtype, precision=precision)
        return codec.decompress_host(np.ascontiguousarray(data[lo:hi]), features=renormalize_features, y_dtype=out_dtype,
                                     precision=precision)
    if world == 1:
        decompressed = run(0, len(data))
    else:  # under torchrun: every rank decodes its contiguous row range, rank 0 collects (the others return None data)
        align = latent_q8.BLOCK_ROWS if quant is not None else 1  # (a quantised latent is cut on its blocks)
        lo, hi = sharded.row_range(len(data), rank, world, align)
        part = run(lo, hi) if hi > lo else np.empty((0, codec.n_features), dtype=out_dtype)
        decompressed = sharded.gather_rows_to_rank0(part, len(data), align=align)
        if decompressed is None:
            return None, names, normalization_features
    if host_renorm is not None:
        decompressed = decompressed * host_renorm[1] + host_renorm[0]
        renormalize_features = host_renorm
    if getattr(config, "save_error_bounded_deltas", False):  # host step; under torchrun rank 0 holds the gathered rows
        decompressed = _apply_deltas(decompressed, input_path_deltas, input_batch_index, int(config.batch_size),
                                     None if renormalize_features is None else renormalize_features[1])
    if conv:
        decompressed = decompressed.reshape(len(decompressed), 1, h, w)
    if config.data_dimension == 2 and config.model_type == "dense":
        decompressed = decompressed.reshape((len(decompressed), original_shape[1], original_shape[2]))
    return decompressed, names, normalization_features
