"""`d3f`-compatible command line (reference: d3f/main.py:6-12).

Commands kept from the reference: `denoise --config --input_list` (d3f/train_denoiser/train_denoiser.py:7-26),
`train new|resume|modify` (d3f/train_deep_fake/start_training.py:8-31).  `sample` is new (BASELINE.json names a
sample entry point the reference does not have; closest reference code: script_tools/put_video_through_fake_model.py).
`balance` is out of scope (SURVEY §2 row 7).  Lightning is replaced by a plain loop; image I/O uses cv2 when the
list file exists, otherwise `--synthetic` feeds seeded low-pass fields (benchmarks / smoke runs)."""
import os

import click
import torch
import yaml

from .train import DeepFakeModule, DenoiserModule, FlatAdam, cosine_lr, set_lr


def read_yaml_file_into_dict(yaml_file_path):
    with open(yaml_file_path) as f:
        return yaml.safe_load(f)


def print_hparams(p):
    print("\nHyper Parameters:")
    for k, v in p.items():
        print(f"\t{k}: {v}")
    print()


def synthetic_batches(batch_size, size, n_batches, device, seed=1234):
    g = torch.Generator(device=device).manual_seed(seed)
    for _ in range(n_batches):
        x = 0.5 * torch.randn(batch_size, 3, size, size, generator=g, device=device)
        yield (torch.nn.functional.avg_pool2d(x, 5, 1, 2) * 2.5).clamp(-1, 1)


def list_file_batches(list_path, batch_size, mean, std, device):
    """Minimal stand-in for d3f/dataset/image_dataset.py + DataLoader: BGR->RGB, (x/255 - mean)/std, NCHW."""
    import cv2
    import numpy as np
    root = os.path.dirname(list_path)
    with open(list_path) as f:
        names = [ln.strip() for ln in f if ln.strip()]
    perm = torch.randperm(len(names)).tolist()
    mean_t = torch.tensor(mean, dtype=torch.float32).view(1, 3, 1, 1)
    std_t = torch.tensor(std, dtype=torch.float32).view(1, 3, 1, 1)
    for i in range(0, len(perm), batch_size):           # the last, smaller batch is kept (DataLoader drop_last=False)
        imgs = []
        for j in perm[i:i + batch_size]:
            img = cv2.cvtColor(cv2.imread(os.path.join(root, names[j])), cv2.COLOR_BGR2RGB)
            imgs.append(torch.from_numpy(np.ascontiguousarray(img)).permute(2, 0, 1).float() / 255.0)
        yield ((torch.stack(imgs) - mean_t) / std_t).to(device, non_blocking=True)


def _optimizers_of(module):
    opts = [getattr(module, n, None) for n in ("optimizer", "optimizer_a", "optimizer_b")]
    return [o for o in opts if o is not None]


def save_checkpoint(path, module, epoch, extra=None):
    """Lightning-shaped checkpoint: {'state_dict', 'hyper_parameters', 'epoch', 'global_step', 'optimizer_states'} with the
    reference's key prefixes (model. / model_a. / model_b. / ema_model_*.ema_model.).  optimizer_states holds the Adam
    moments, step count and current LR of every optimiser (Lightning's `ckpt_path` resume restores them,
    d3f/train_deep_fake/start_training.py:19-23, :50-53)."""
    ckpt = {"state_dict": module.state_dict(), "hyper_parameters": dict(module.hparams), "epoch": epoch,
            "global_step": module.global_step,
            "optimizer_states": [o.state_dict() for o in _optimizers_of(module)]}
    ckpt.update(extra or {})
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    torch.save(ckpt, path)


def load_checkpoint(path, cls, strict=True, **overrides):
    ckpt = torch.load(path, map_location="cpu", weights_only=False)
    hp = dict(ckpt["hyper_parameters"])
    hp.update(overrides)
    module = cls(**hp)
    module.load_state_dict(ckpt["state_dict"], strict=strict)
    module.current_epoch = ckpt.get("epoch", 0)
    module.global_step = ckpt.get("global_step", 0)
    return module, ckpt


def restore_optimizers(module, ckpt):
    """After configure_optimizers(): Adam moments / step counts from the checkpoint (when the optimiser form matches) and the
    cosine LR of the epoch being resumed — a resumed run continues at cosine_lr(current_epoch), not at the base LR."""
    states = ckpt.get("optimizer_states") or []
    opts = _optimizers_of(module)
    if len(states) == len(opts):
        for o, sd in zip(opts, states):
            if isinstance(o, FlatAdam) == ("m" in sd and "v" in sd):
                if isinstance(o, FlatAdam):
                    o.load_state_dict({k: (v.to(o.m.device) if torch.is_tensor(v) else v) for k, v in sd.items()})
                else:
                    o.load_state_dict(sd)
    p = module.hparams
    lr = cosine_lr(p["learning_rate"], module.current_epoch, p["cosine_scheduler_max_epoch"])
    for o in opts:
        set_lr(o, lr)


@click.group()
def cli():
    pass


@cli.command()
@click.option("--config", required=True, help="Path to config yaml file")
@click.option("--input_list", required=False, default=None, help="Text file listing relative image paths")
@click.option("--synthetic", type=int, default=0, help="Use N synthetic batches per epoch instead of --input_list")
@click.option("--size", type=int, default=64)
@click.option("--precision", default="bf16", type=click.Choice(["bf16", "fp32"]))
@click.option("--checkpoint_dir", default="d3fk_checkpoints")
def denoise(config, input_list, synthetic, size, precision, checkpoint_dir):
    """Train the denoiser (reference: `d3f denoise`)."""
    if not input_list and not synthetic:
        raise click.UsageError("give --input_list (the reference's image list) or --synthetic N (seeded synthetic batches)")
    hp = read_yaml_file_into_dict(config)
    hp["input_image_list_path"] = input_list
    hp.setdefault("precision", precision)
    # the reference's training step always runs its kornia RandomAffine on the batch (lit_module.py:55-65, :113); here it is
    # fused with the noising (d3fk_affine_q_sample).  `augment: false` in the YAML turns it off.
    hp.setdefault("augment", True)
    dev = torch.device("cuda", torch.cuda.current_device())
    module = DenoiserModule(**hp).to(dev).train()
    print_hparams(module.hparams)
    module.configure_optimizers(fused=True)
    mean = [m / 255.0 for m in hp.get("mean", [127.5] * 3)]
    std = [s / 255.0 for s in hp.get("std", [127.5] * 3)]
    for epoch in range(hp["max_epochs"]):
        batches = (synthetic_batches(hp["batch_size"], size, synthetic, dev, seed=epoch) if synthetic
                   else list_file_batches(input_list, hp["batch_size"], mean, std, dev))
        for image in batches:
            loss = module.training_step(image)
        module.on_epoch_end()
        print(f"epoch {epoch} loss {float(loss):.5f} lr {module.optimizer.lr:.3g}")
        save_checkpoint(os.path.join(checkpoint_dir, "last.ckpt"), module, epoch + 1)


def _fit_deep_fake(module, size, synthetic, checkpoint_dir, ckpt=None):
    p = module.hparams
    dev = torch.device("cuda", torch.cuda.current_device())
    module.to(dev).train()
    if not synthetic:
        p.setdefault("augment", True)      # list-file data: the reference's ShiftScaleRotate (lit_module.py:99-111)
    print_hparams(p)
    module.configure_optimizers()
    if ckpt is not None:
        restore_optimizers(module, ckpt)
    for epoch in range(module.current_epoch, p["max_epochs"]):
        if synthetic:
            it = zip(synthetic_batches(p["batch_size"], size, synthetic, dev, seed=2 * epoch),
                     synthetic_batches(p["batch_size"], size, synthetic, dev, seed=2 * epoch + 1))
        else:
            it = zip(list_file_batches(p["data_path_a"], p["batch_size"], p["mean_a"], p["std_a"], dev),
                     list_file_batches(p["data_path_b"], p["batch_size"], p["mean_b"], p["std_b"], dev))
        for batch_a, batch_b in it:
            module.training_step(batch_a, batch_b)
        module.on_epoch_end()
        print(f"epoch {epoch} " + " ".join(f"{k}={float(v):.5f}" for k, v in module.logged.items()))
        save_checkpoint(os.path.join(checkpoint_dir, "last.ckpt"), module, epoch + 1)


@cli.group()
def train():
    """Train the two-identity deep-fake model (reference: `d3f train new|resume|modify`)."""


_common = [click.option("--synthetic", type=int, default=0), click.option("--size", type=int, default=128),
           click.option("--checkpoint_dir", default="d3fk_checkpoints")]


def _add(opts):
    def deco(f):
        for o in reversed(opts):
            f = o(f)
        return f
    return deco


@train.command()
@click.option("--config_path", required=True, help="Path to the config yaml.")
@_add(_common)
def new(config_path, synthetic, size, checkpoint_dir):
    module = DeepFakeModule(**read_yaml_file_into_dict(config_path))
    _fit_deep_fake(module, size, synthetic, checkpoint_dir)


@train.command()
@click.option("--checkpoint_path", required=True, help="Path to model checkpoint.")
@_add(_common)
def resume(checkpoint_path, synthetic, size, checkpoint_dir):
    module, ckpt = load_checkpoint(checkpoint_path, DeepFakeModule)
    _fit_deep_fake(module, size, synthetic, checkpoint_dir, ckpt)


@train.command()
@click.option("--config_path", required=True, help="Path to the config yaml.")
@click.option("--checkpoint_path", required=True, help="Path to model checkpoint.")
@_add(_common)
def modify(config_path, checkpoint_path, synthetic, size, checkpoint_dir):
    """Load weights non-strictly and overlay new hyper-parameters (denoise -> swap stage hand-over)."""
    module, _ = load_checkpoint(checkpoint_path, DeepFakeModule, strict=False, **read_yaml_file_into_dict(config_path))
    module.current_epoch = 0
    _fit_deep_fake(module, size, synthetic, checkpoint_dir)


@cli.command()
@click.option("--checkpoint_path", default=None, help="Denoiser or deep-fake checkpoint (random init if omitted)")
@click.option("--model", "which", default="a", type=click.Choice(["a", "b", "denoiser"]))
@click.option("--steps", type=int, default=50)
@click.option("--batch", type=int, default=8)
@click.option("--size", type=int, default=64)
@click.option("--eta", type=float, default=1.0, help="0 = DDIM, 1 = DDPM ancestral")
@click.option("--r_start", type=float, default=1.0, help="noise ratio to start from (1 = pure noise)")
@click.option("--seed", type=int, default=0)
@click.option("--out", default="samples.pt")
@click.option("--source", default=None, help="torch.save'd normalised images [B,3,H,W] to inpaint (needs --mask; "
              "sets the batch and size)")
@click.option("--mask", default=None, help="torch.save'd mask [H,W], [1,1,H,W] or [B,1,H,W]: 1 = generate, 0 = keep "
              "the source, fractions feather")
@click.option("--solver", default="posterior", type=click.Choice(["posterior", "dpmpp-2m"]),
              help="posterior = first-order update; dpmpp-2m = second-order multistep DPM-Solver++ 2M")
@click.option("--schedule", default=None, type=click.Choice(["linear", "logsnr"]),
              help="noise-ratio grid (default: linear for posterior, logsnr for dpmpp-2m)")
def sample(checkpoint_path, which, steps, batch, size, eta, r_start, seed, out, source, mask, solver, schedule):
    """Iterative reverse-diffusion sampling with CUDA-graph replayed steps (new entry point).  With --source and --mask
    the sampler regenerates only the masked region and keeps the source outside it (masked face swap)."""
    from .sampler import Sampler
    from .unet import Unet
    if (source is None) != (mask is None):
        raise click.UsageError("--source and --mask go together")
    dev = torch.device("cuda", torch.cuda.current_device())
    if checkpoint_path:
        try:
            module, _ = load_checkpoint(checkpoint_path, DenoiserModule)
            model = module.model
        except Exception:
            module, _ = load_checkpoint(checkpoint_path, DeepFakeModule)
            model = module.model_a if which == "a" else module.model_b
    else:
        model = Unet()
    model = model.to(dev).eval()
    method = dict(solver=solver.replace("-", "_"), schedule=schedule)
    if source is None:
        smp = Sampler(model, batch, size, size, steps, r_start=r_start, eta=eta, seed=seed, **method)
        x0 = smp.run()
    else:
        src = torch.load(source, map_location="cpu").to(dev, torch.float32).contiguous()
        if src.dim() != 4 or src.shape[1] != 3:
            raise click.UsageError(f"--source must hold [B,3,H,W] images, got {tuple(src.shape)}")
        B, _, H, W = src.shape
        smp = Sampler(model, B, H, W, steps, r_start=r_start, eta=eta, seed=seed, masked=True, **method)
        x0 = smp.run(src=src, mask=torch.load(mask, map_location="cpu"))
    torch.save(x0.cpu(), out)
    print(f"wrote {tuple(x0.shape)} samples to {out}")


if __name__ == "__main__":
    cli()
