"""Training / evaluation drivers -- mirror of /root/reference/scripts/runners.py: `create_dataset` (:21-62),
`create_model` (:65-103), `run_train` (:106-232), `run_eval` (:235-458).  Host side only: the step, the
forward-only helpers and the binarisation of the input run in the native library.

Differences from the reference, all forced by asynchronous execution or by what this image lacks:
* data: local MNIST files (`--dataset_path` / $GMVAE_MNIST_DIR; IDX or mnist.npz) or a synthetic stand-in
  instead of TFDS; intensities stay in HBM and are binarised on the device (data.py).
* the loss is read back once per `summarise_every` steps (one device->host sync) together with the
  per-step losses of that window, and the early-stopping hook is then replayed over every step: the rule
  and its step counts are the reference's (utils.py:13-57); the stop is noticed at most
  `summarise_every - 1` steps late.
* summaries are `summaries.jsonl` + PNG tiles instead of TF event files; plots are plain rasters
  (matplotlib / seaborn are absent); checkpoints are torch files with the reference's variable names
  in the Saver's `model.ckpt-<step>` + `checkpoint` layout.
* one process per GPU under torchrun splits every global batch of `world * batch_size` rows by rank
  (the reference is single-device, :193)."""
from __future__ import annotations

import os
import sys
import time
from typing import Optional

import numpy as np
import torch

from . import data as data_mod
from . import dist as dist_mod
from . import gmvae as gmvae_mod
from . import utils
from . import vae as vae_mod

IMG_SHAPE = data_mod.IMG_SHAPE


class _ShapedBatches:
    """Iterator adaptor giving the reference's tensor contract: images [B, 28, 28, 1] (uint8 {0,1} on the device,
    the reference's bool), labels int64 [B] (runners.py:32-35)."""

    def __init__(self, dataset: data_mod.DeviceDataset, shape=IMG_SHAPE):
        self.dataset, self.shape = dataset, shape
        self._it = None

    def __iter__(self):
        self._it = iter(self.dataset)
        return self

    def __next__(self):
        if self._it is None:
            self._it = iter(self.dataset)
        x, labels = next(self._it)
        return x.reshape(x.shape[0], *self.shape), labels

    @property
    def last_global_rows(self) -> int:
        return self.dataset.last_global_rows

    @property
    def num_examples(self) -> int:
        return self.dataset.num_examples


def create_dataset(config, split: str, shuffle: bool, repeat: bool, engine=None, world: int = 1, rank: int = 0,
                   first_draw: int = 0):
    """runners.py:21-62.  `engine` supplies the device and `Engine.binarize`; `config.batch_size` is the
    per-device batch, so a global batch holds `world * batch_size` rows."""
    if engine is None:
        raise RuntimeError("create_dataset needs the model's engine: the input is binarised on the device (no CPU fallback)")
    path = getattr(config, "dataset_path", None) or os.environ.get("GMVAE_MNIST_DIR")
    loaded = data_mod.load_mnist(path, split)
    if loaded is None:
        if path:
            raise FileNotFoundError(f"no MNIST files (IDX or mnist.npz) for split {split!r} under {path}")
        loaded = data_mod.synthetic_mnist(split, data_size=engine.data_size)
    images, labels = loaded
    dev = engine.device
    ds = data_mod.DeviceDataset(torch.from_numpy(images).to(dev), torch.from_numpy(labels).to(dev),
                                batch_size=config.batch_size * world, shuffle=shuffle, repeat=repeat,
                                binarize=engine.binarize, seed=getattr(config, "random_seed", None) or 0,
                                first_draw=first_draw, world=world, rank=rank)
    return _ShapedBatches(ds)


def create_model(config, data_dim: int):
    """runners.py:65-103: the hyper-parameters that are not flags are fixed here exactly as there."""
    hidden = [config.hidden_size] * config.num_layers
    if config.model == "gmvae":
        model = gmvae_mod.create_gmvae(data_dim, config.latent_size, mixture_components=config.mixture_components,
                                       fcnet_hidden_sizes=hidden, sigma_min=0.0, raw_sigma_bias=0.5, temperature=1.0)
    elif config.model == "vae_gmp":
        model = vae_mod.create_vae(data_dim, config.latent_size, mixture_components=config.mixture_components,
                                   fcnet_hidden_sizes=hidden, sigma_min=0.0, raw_sigma_bias=0.5)
    else:
        model = vae_mod.create_vae(data_dim, config.latent_size, fcnet_hidden_sizes=hidden, sigma_min=0.0, raw_sigma_bias=0.5)
    return model


def logdir_for(config) -> str:
    """runners.py:212-217."""
    return "{}/{}/h{}_n{}_z{}".format(config.logdir, config.model, config.hidden_size, config.num_layers, config.latent_size)


def _configure(model, config, device: int):
    model.configure(precision=getattr(config, "precision", "bf16"), objective=getattr(config, "objective", "reference"),
                    learning_rate=getattr(config, "learning_rate", 1e-3), max_batch=config.batch_size, device=device,
                    deterministic=getattr(config, "deterministic", False))
    model.random_seed = config.random_seed
    return model.engine(config.batch_size)


def _device_of(config) -> int:
    return int(config.gpu_id) if str(config.gpu_id).isdigit() else 0


def write_image_summaries(writer: utils.SummaryWriter, model, config, images, flat_inputs, step: int):
    """The `image_summaries` scope of create_model_loss (runners.py:132-157): 5x5 inputs, 5x5 reconstructions,
    3x3 decoded prior samples (one per component for the GMVAE, ten for the VAEs)."""
    utils.image_tile_summary(writer, "inputs", images.float(), step, rows=5, cols=5)
    recon = utils.unflatten_tensor(model.reconstruct_images(flat_inputs), IMG_SHAPE)
    utils.image_tile_summary(writer, "reconstructions", recon, step, rows=5, cols=5)
    sampled_z = model.generate_samples(num_samples=1 if config.model == "gmvae" else 10)
    samples = utils.unflatten_tensor(model.generate_sample_images(z=sampled_z), IMG_SHAPE)
    utils.image_tile_summary(writer, "samples", samples, step, rows=3, cols=3)


def run_train(config):
    """runners.py:106-232."""
    world, rank, local = dist_mod.env_world()
    if world > 1:
        dist_mod.init_process_group("nccl")
    torch.manual_seed(config.random_seed or 0)
    model = create_model(config, data_dim=int(np.prod(IMG_SHAPE)))
    eng = _configure(model, config, local if world > 1 else _device_of(config))
    if world > 1:
        eng.init_data_parallel()
    logdir = logdir_for(config)
    if not os.path.exists(logdir):
        if rank == 0:
            print("Creating log directory at {}".format(logdir))
        os.makedirs(logdir, exist_ok=True)
    if utils.restore_checkpoint_if_exists(eng, logdir) and rank == 0:  # MonitoredTrainingSession auto-restore (:222-225)
        print(f"Restored checkpoint of step {eng.global_step} from {logdir}")
    cur_step = eng.global_step
    batches = create_dataset(config, "train", shuffle=True, repeat=True, engine=eng, world=world, rank=rank,
                             first_draw=cur_step)             # new uniforms after a resume, too
    hook = utils.EarlyStoppingHook(max_steps=config.early_stop_rounds, threshold=config.early_stop_threshold)
    writer = utils.SummaryWriter(logdir) if rank == 0 else None
    every = max(1, int(config.summarise_every))
    history = torch.zeros(every, 4, dtype=torch.float32, device=eng.device)   # per-step loss terms of the current window
    pending = 0
    last_save, t0 = time.time(), time.time()
    while not hook.stop_requested and cur_step <= config.max_steps:
        images, labels = next(batches)
        flat_inputs = utils.flatten_tensor(images, IMG_SHAPE)
        loss = eng.train_step(flat_inputs, global_batch=batches.last_global_rows)
        cur_step += 1
        history[pending].copy_(loss, non_blocking=True)
        pending += 1
        if pending == every or cur_step > config.max_steps:
            window = history[:pending].cpu()                           # the only device->host sync of the loop
            for i in range(pending):
                hook.after_run(float(window[i, 0]), cur_step - pending + 1 + i)
            t = window[pending - 1].tolist()
            if rank == 0:
                print(utils.summary_formatter({"step": cur_step, "loss": t[0]}), flush=True)
                rec = {"elbo": -t[0], "nll_scalar": t[1], "kl_div_z": t[2],
                       "global_step/sec": pending / max(time.time() - t0, 1e-9)}
                if config.model == "gmvae":
                    rec["nent"] = t[3]
                    rec["cluster_acc"] = utils.cluster_acc(model.encoder_y_logits(flat_inputs), labels,
                                                           config.mixture_components)      # gmvae.py:270-272
                writer.scalars(cur_step, rec)
                if getattr(config, "image_summaries", 1):
                    write_image_summaries(writer, model, config, images, flat_inputs, cur_step)
            pending, t0 = 0, time.time()
        if rank == 0 and time.time() - last_save > 120:                # save_checkpoint_secs=120 (:226)
            utils.save_checkpoint(eng.state_dict(), logdir, cur_step)
            last_save = time.time()
    if rank == 0:
        utils.save_checkpoint(eng.state_dict(), logdir, cur_step)
        writer.close()
    return eng


def process_over_dataset(model, eng, batches, config):
    """runners.py:301-337.  Returns (avg_loss, corrected, latent_state, labels): `avg_loss` is the reference's number --
    it adds up the per-batch *mean* losses (`tf.reduce_sum` of a scalar, :298) and divides by the number of
    examples (:335), i.e. it is ~1/batch_size of the per-example loss (SURVEY F10) -- and `corrected` is the
    example-weighted mean loss that was meant."""
    total_loss, total_n_elems, weighted = 0.0, 0.0, 0.0
    latent_state, labels_out = [], []
    for images, labels in batches:
        flat_inputs = utils.flatten_tensor(images, IMG_SHAPE)
        bs = flat_inputs.shape[0]
        z = model.transform(flat_inputs)
        loss = float(model.run_model(flat_inputs, flat_inputs, labels) if config.model == "gmvae"
                     else model.run_model(flat_inputs, flat_inputs))
        total_loss += loss
        weighted += loss * bs
        total_n_elems += bs
        latent_state.extend(z.cpu().numpy().reshape(-1, config.latent_size))
        labels_out.extend(labels.cpu().numpy().reshape(-1, 1))
    n = max(total_n_elems, 1.0)
    return total_loss / n, weighted / n, np.array(latent_state), np.array(labels_out)


def run_eval(config, max_wait: Optional[float] = None):
    """runners.py:235-458: one pass over `config.split`, loss summary, latent / prior-sample plots, image grids."""
    torch.manual_seed(config.random_seed or 0)
    if config.random_seed:
        np.random.seed(config.random_seed)
    model = create_model(config, data_dim=int(np.prod(IMG_SHAPE)))
    eng = _configure(model, config, _device_of(config))
    logdir = logdir_for(config)
    if not os.path.exists(logdir):
        print("No directory {}".format(logdir), file=sys.stderr)
        sys.exit(1)
    summary_dir = "{}/{}".format(logdir, config.split)
    writer = utils.SummaryWriter(summary_dir)
    utils.wait_for_checkpoint(eng, logdir, max_wait=max_wait)
    step = eng.global_step
    print("Model restored from step %d" % step)

    batches = create_dataset(config, config.split, shuffle=False, repeat=False, engine=eng)
    avg_loss, corrected, z_out, y_out = process_over_dataset(model, eng, batches, config)
    writer.scalars(step, {"%s/loss_per_example" % config.split: avg_loss,
                          "%s/loss_per_example_corrected" % config.split: corrected})
    print("%s loss/example: %f" % (config.split, avg_loss))

    print("Plotting latent code!")
    z_two = utils.reduce_dimensionality(z_out, random_state=config.random_seed)
    utils.scatter_png("{}/step_{}".format(summary_dir, step), z_two, y_out, n_classes=config.mixture_components)

    samples = model.generate_samples(num_samples=config.num_samples)
    sample_images = utils.unflatten_tensor(model.generate_sample_images(num_samples=config.num_generations), IMG_SHAPE)
    print("Plotting prior samples!")
    samples_two = utils.reduce_dimensionality(samples, random_state=config.random_seed)
    utils.scatter_png("{}/step_{}_samples".format(summary_dir, step), samples_two)
    utils.display_images("{}/step_{}_sample_images".format(summary_dir, step), sample_images)
    if config.model == "gmvae":
        k = int(np.random.randint(0, high=config.mixture_components))
        samples_k = model.generate_samples(num_samples=config.num_generations * config.mixture_components, clusters=[k])
        sample_images_k = utils.unflatten_tensor(model.generate_sample_images(samples_k, name="sample_images_k"), IMG_SHAPE)
        utils.display_images("{}/step_{}_sample_k_images".format(summary_dir, step), sample_images_k)
    writer.close()
    return {"step": step, "avg_loss": avg_loss, "loss_per_example": corrected, "z": z_out, "labels": y_out,
            "summary_dir": summary_dir}
