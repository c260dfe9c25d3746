"""Command line -- same flags, defaults and `--flag=value` syntax as
/root/reference/scripts/run_gmvae.py:11-58 (tf.app.flags), plus additive flags (`--precision`,
`--objective`, `--dataset_path`, `--image_summaries`, `--deterministic`).  Data parallelism needs no flag: launch with
`torchrun --nproc-per-node N -m gmvae_b200.run_gmvae ...` and `--batch_size` is the per-GPU batch.

    python -m gmvae_b200.run_gmvae --mode=train --model=gmvae --latent_size=64 --hidden_size=512 \
        --num_layers=2 --batch_size=100 --max_steps=200
"""
from __future__ import annotations

import argparse

from . import runners


def build_parser() -> argparse.ArgumentParser:
    p = argparse.ArgumentParser(description="GMVAE / VAE training on B200")
    # Shared flags (run_gmvae.py:11-31)
    p.add_argument("--mode", default="train", choices=["train", "eval"], help="The mode of the binary.")
    p.add_argument("--model", default="gmvae", choices=["gmvae", "vae", "vae_gmp"], help="Model choice.")
    p.add_argument("--latent_size", type=int, default=8, help="Number of dimensions in the latent state.")
    p.add_argument("--hidden_size", type=int, default=64, help="Number of dimensions in the hidden layers.")
    p.add_argument("--num_layers", type=int, default=1, help="Number of hidden layers in the internal networks.")
    p.add_argument("--mixture_components", type=int, default=10, help="Number of mixture components.")
    p.add_argument("--batch_size", type=int, default=16, help="Batch size.")
    p.add_argument("--logdir", default="/tmp/smc_vi", help="The directory to keep checkpoints and summaries in.")
    p.add_argument("--random_seed", type=int, default=None, help="A random seed.")
    # Training flags (run_gmvae.py:35-48)
    p.add_argument("--learning_rate", type=float, default=0.001, help="The learning rate for ADAM.")
    p.add_argument("--max_steps", type=int, default=int(1e9), help="The number of gradient update steps to train for.")
    p.add_argument("--early_stop_rounds", type=int, default=1000, help="Steps before terminating due to early stopping.")
    p.add_argument("--early_stop_threshold", type=float, default=0.001, help="Early stopping threshold.")
    p.add_argument("--summarise_every", type=int, default=50, help="The number of steps between summaries.")
    p.add_argument("--gpu_id", default="0", help="GPU device id to use.")
    p.add_argument("--gpu_num", default="0", help="Comma-separated list of GPU ids to use.")
    # Evaluation flags (run_gmvae.py:52-58)
    p.add_argument("--num_samples", type=int, default=10, help="Number of samples to draw from a model's prior.")
    p.add_argument("--num_generations", type=int, default=10, help="Number of generated images to yield.")
    p.add_argument("--split", default="train", choices=["train", "test"], help="Split to evaluate the model on.")
    # Additive flags (no reference counterpart)
    p.add_argument("--precision", default="bf16", choices=["bf16", "fp32"], help="GEMM path: tcgen05 bf16 or fp32 validation.")
    p.add_argument("--objective", default="reference", choices=["reference", "marginal"], help="See DESIGN.md section 1.")
    p.add_argument("--dataset_path", default=None, help="Directory with the MNIST IDX files (plain or .gz) or mnist.npz; "
                   "default $GMVAE_MNIST_DIR, else a synthetic stand-in (the reference downloads through TFDS).")
    p.add_argument("--image_summaries", type=int, default=1, help="Write the input / reconstruction / sample tiles with "
                   "every summary (the reference always does).")
    p.add_argument("--deterministic", action="store_true", help="Bitwise-reproducible training steps: the same seed, data and "
                   "configuration give identical parameters (slower; DESIGN.md section 9).")
    return p


def main(argv=None):
    flags = build_parser().parse_args(argv)
    if flags.mode == "train":
        runners.run_train(flags)
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():         # torchrun: leave together
            dist.barrier()
            dist.destroy_process_group()
    elif flags.mode == "eval":
        runners.run_eval(flags)


if __name__ == "__main__":
    main()
