"""The reference's validation / inference loop (sr_mfe.py:258-386, infer.py:62-119) on the B200 path:
batched LR images -> bit-exact bicubic conditioning -> T-step sampling -> device-side MSE / PSNR / SSIM /
ERGAS against HR (for both the bicubic baseline 'INF' and the SR result), averaged like the reference.

Differences, all deliberate: images are processed in batches (the reference feeds one image per step and
crashes for B>1, SURVEY F2); metrics are computed on the device (`fdsr_metrics_u8`, or `fdsr_metrics_u16` at the
white level of 16-bit data) instead of skimage +
matplotlib on the host; LPIPS (an AlexNet download) and the per-image matplotlib plot are not produced;
under torchrun the dataset is sharded by image and the sums are all-reduced, or, with `tile_split`, every rank samples
every image together with the others (each its share of the tiles) and the metrics are counted once.
"""
from __future__ import annotations

import logging
import os
import time

import numpy as np
import torch
import torch.distributed as dist

from .data import BatchLoader, nodata_mask, u16_to_tensor, u8_to_tensor
from .parallel import reduce_sums, shard_bounds

METRIC_NAMES = ("mse", "psnr", "ssim", "ergas")


def load_network(netG, opt, logger=None):
    """model/model.py:148-160: `{resume_state}_gen.pth`, strict unless finetune_norm."""
    load_path = opt['path']['resume_state'] if opt['path'] is not None else None
    if load_path is None:
        return False
    gen_path = '{}_gen.pth'.format(load_path)
    if not os.path.exists(gen_path):
        raise FileNotFoundError(f"checkpoint {gen_path} not found (path.resume_state of the config)")
    if logger:
        logger.info('Loading pretrained model for G [{:s}] ...'.format(load_path))
    sd = torch.load(gen_path, map_location="cpu")
    # The reference saves netG.state_dict() after set_new_noise_schedule (model/model.py:126-146), so a real
    # `*_gen.pth` carries the 12 schedule buffers.  They load strictly when the schedule has been registered first
    # (the reference's order, model/model.py:19-41, which `main` follows); a netG without them gets the denoiser only.
    own = set(netG.state_dict().keys())
    from .diffusion import _BUFFERS
    sd = {k: v for k, v in sd.items() if not (k in _BUFFERS and k not in own)}
    netG.load_state_dict(sd, strict=(not opt['model']['finetune_norm']))
    return True


def _fill(img_hwc, fill):
    """fill = (valid (H,W) bool tensor, V): every band of the invalid pixels set to V, in place."""
    if fill is not None:
        img_hwc[~fill[0].cpu().numpy()] = fill[1]
    return img_hwc


def _save_u8(img_chw, path, fill=None):
    """RGB for 3 bands, a single-band 'L' image for 1, an (H,W,C) uint8 `.npy` array (extension replaced) otherwise.
    `fill` = (valid, V): the invalid pixels are written as V in every band.  Returns the path written."""
    from PIL import Image
    a = img_chw.detach().float().clamp(-1, 1)
    a = ((a + 1) / 2).permute(1, 2, 0).cpu().numpy()
    u8 = _fill((a * 255.0).round().astype(np.uint8), fill)
    if u8.shape[2] == 3:
        Image.fromarray(u8).save(path)
    elif u8.shape[2] == 1:
        Image.fromarray(u8[:, :, 0]).save(path)  # 2-D uint8: mode L
    else:
        path = os.path.splitext(path)[0] + ".npy"
        np.save(path, u8)
    return path


def _save_u16(img_chw, path, max_value, fill=None):
    """The 16-bit tensor2img at white level M = max_value, rint(((clamp(x,-1,1) + 1) / 2) * M) in fp32 (ties to even),
    saved as a single-band I;16 image (PNG / TIFF) for 1 band and as an (H,W,C) uint16 `.npy` array (extension replaced)
    for any other band count, 3 included.  `fill` = (valid, V): the invalid pixels are written as V in every band.
    Returns the path written."""
    from PIL import Image
    a = img_chw.detach().float().clamp(-1, 1)
    a = ((a + 1) / 2).permute(1, 2, 0).cpu().numpy()
    u16 = _fill((a * np.float32(max_value)).round().astype(np.uint16), fill)
    if u16.shape[2] == 1:
        Image.fromarray(u16[:, :, 0]).save(path)  # 2-D uint16: mode I;16
    else:
        path = os.path.splitext(path)[0] + ".npy"
        np.save(path, u16)
    return path


@torch.no_grad()
def evaluate(netG, dataset, batch_size=16, scale=4, result_path=None, save_ext="tif", seed=0, current_step=0,
             logger=None, max_images=None, tile=None, tile_overlap=32, tile_batch=16, tile_split=False):
    """Returns {'n', 'bic_mse', 'bic_psnr', 'bic_ssim', 'bic_ergas', 'sr_mse', ..., 'seconds', 'images_per_s'}.
    `tile`: sample every image as one canvas of overlapping tiles (GaussianDiffusion.super_resolution(tile=...)), one
    image per call (scenes may differ in size; the tiles of one canvas fill the GPU); the HR size is then `scale` x the
    LR size, whatever that size is.  `tile_split` (with `tile`, under torchrun): the ranks split each image's tiles
    instead of sharding the images (GaussianDiffusion.super_resolution(tile_split=True)); rank 0 writes the images.
    A 16-bit dataset (`dataset.max_value` = M) is conditioned by `fdsr_bicubic_u16` (or its sr_ folder through
    u16_to_tensor), scored by `fdsr_metrics_u16` at M and saved as 16-bit images; the returned keys are the same.
    A dataset with a fill value (`dataset.nodata` = V) is scored on its valid pixels (nodata_mask of the LR image, or
    of the sr_ image without LR; fdsr_metrics_masked), tiled sampling skips the tiles with no valid pixel, every band of
    an invalid pixel is written as V, and an image whose eight metrics are not all finite (no valid pixel, or no wholly
    valid SSIM window) is left out of the averages; 'n_excluded' counts those."""
    if tile_split and tile is None:
        raise ValueError("tile_split needs tile")
    if tile is not None:
        batch_size = 1
    tiling = {} if tile is None else dict(tile=tile, tile_overlap=tile_overlap, tile_batch=tile_batch,
                                          tile_split=tile_split)
    eng = netG.engine()
    dev = eng.device
    world = dist.get_world_size() if dist.is_initialized() else 1
    rank = dist.get_rank() if dist.is_initialized() else 0
    n_total = len(dataset) if max_images is None else min(len(dataset), max_images)
    # tile_split: every rank holds every image's result, so the images are not sharded and the sums not reduced
    start, stop, _ = (0, n_total, n_total) if tile_split else shard_bounds(n_total, rank, world)
    write = result_path and (rank == 0 or not tile_split)
    loader = BatchLoader(dataset, batch_size, indices=range(start, stop))
    acc = torch.zeros(10, dtype=torch.float64, device=dev)      # bic[4], sr[4], n averaged, n excluded
    M = getattr(dataset, "max_value", None)                      # None: 8-bit data
    nodata = getattr(dataset, "nodata", None)                    # None: every pixel is valid
    if M is None:
        to_tensor, metrics, save = u8_to_tensor, eng.metrics_u8, _save_u8
    else:
        to_tensor = lambda x: u16_to_tensor(x, M)                                  # noqa: E731
        metrics = lambda a, b, s, valid=None: eng.metrics_u16(a, b, M, s, valid)   # noqa: E731
        save = lambda img, path, fill=None: _save_u16(img, path, M, fill)          # noqa: E731
    if write:                        # every rank writes its own shard's images there (tile_split: rank 0 all of them)
        os.makedirs(result_path, exist_ok=True)
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for bi, batch in enumerate(loader):
        hr = to_tensor(batch["HR"].to(dev, non_blocking=True))
        H, W = hr.shape[2], hr.shape[3]
        if tile is not None and "LR" in batch:
            H, W = scale * batch["LR"].shape[1], scale * batch["LR"].shape[2]
            if (hr.shape[2], hr.shape[3]) != (H, W):
                raise ValueError(f"image {batch['Index'][0]}: HR is {hr.shape[2]}x{hr.shape[3]}, not {scale} x the LR "
                                 f"size ({H}x{W})")
        valid = None
        if nodata is not None:                                     # the footprint: from LR, else from the sr_ image
            valid = nodata_mask(batch["LR" if "LR" in batch else "SR"].to(dev, non_blocking=True), nodata, H, W)
        if "SR" in batch:                                          # the reference's precomputed bicubic image
            cond = to_tensor(batch["SR"].to(dev, non_blocking=True)).contiguous()
        elif M is None:
            _, cond = eng.bicubic_u8(batch["LR"].to(dev, non_blocking=True), H, W, want_u8=False)
        else:
            _, cond = eng.bicubic_u16(batch["LR"].to(dev, non_blocking=True), H, W, M, want_u16=False)
        # one seed for the whole job; the noise of an image depends on its global dataset index only, so the result
        # does not depend on the batch size or the number of ranks
        masked = {} if valid is None or tile is None else {"valid": valid}   # untiled: every pixel is sampled
        sr = netG.super_resolution(cond, False, seed=seed, image_offset=start + bi * loader.bs, **tiling, **masked)
        if sr.dim() == 3:   # the SR3 baseline returns ret_img[-1] without the batch axis for a single image
            sr = sr[None]
        if valid is None:
            m_bic = metrics(cond, hr, scale)
            m_sr = metrics(sr, hr, scale)
            acc[0:4] += m_bic.sum(0)
            acc[4:8] += m_sr.sum(0)
            acc[8] += hr.shape[0]
        else:
            m_bic = metrics(cond, hr, scale, valid=valid)
            m_sr = metrics(sr, hr, scale, valid=valid)
            keep = torch.isfinite(m_bic).all(1) & torch.isfinite(m_sr).all(1)
            acc[0:4] += m_bic[keep].sum(0)
            acc[4:8] += m_sr[keep].sum(0)
            acc[8] += keep.sum()
            acc[9] += (~keep).sum()
        if write:
            for j, idx in enumerate(batch["Index"]):
                fill = None if valid is None else (valid[j], nodata)
                save(sr[j], '{}/{}_{}_sr.{}'.format(result_path, current_step, idx + 1, save_ext), fill=fill)
    torch.cuda.synchronize(dev)
    dt = time.perf_counter() - t0
    if not tile_split:
        reduce_sums(acc)
    n = max(acc[8].item(), 1.0)
    n_all = acc[8].item() + acc[9].item()
    out = {"n": int(n_all), "seconds": dt, "images_per_s": n_all / dt if dt > 0 else float("nan")}
    if nodata is not None:
        out["n_excluded"] = int(acc[9].item())
    for i, k in enumerate(METRIC_NAMES):
        out["bic_" + k] = acc[i].item() / n
        out["sr_" + k] = acc[4 + i].item() / n
    if logger and rank == 0:
        logger.info('bic_mse: {:.5e}, bic_psnr: {:.5e}, bic_ssim：{:.5e}, bic_ergas: {:.5e}'.format(
            out["bic_mse"], out["bic_psnr"], out["bic_ssim"], out["bic_ergas"]))
        logger.info('sr_mse: {:.5e}, sr_psnr: {:.5e}, sr_ssim：{:.5e}, sr_ergas: {:.5e}'.format(
            out["sr_mse"], out["sr_psnr"], out["sr_ssim"], out["sr_ergas"]))
        logger.info('{} images in {:.3f} s ({:.1f} images/s, batch {} x {} rank(s))'.format(
            out["n"], dt, out["images_per_s"], batch_size, world))
        if nodata is not None:
            logger.info('nodata {}: {} image(s) without a finite score left out of the averages'.format(
                nodata, out["n_excluded"]))
    return out


def setup_logger(name="base", log_dir=None, screen=True):
    lg = logging.getLogger(name)
    if lg.handlers:
        return lg
    lg.setLevel(logging.INFO)
    fmt = logging.Formatter('%(asctime)s.%(msecs)03d - %(levelname)s: %(message)s', datefmt='%y-%m-%d %H:%M:%S')
    if log_dir:
        os.makedirs(log_dir, exist_ok=True)
        fh = logging.FileHandler(os.path.join(log_dir, name + ".log"), mode="w")
        fh.setFormatter(fmt)
        lg.addHandler(fh)
    if screen:
        sh = logging.StreamHandler()
        sh.setFormatter(fmt)
        lg.addHandler(sh)
    return lg


def parse_args(argv=None, default_config="config/sr_fastdiffsr_test_64_256.json", prog="sr_mfe.py"):
    """The flags of the repo-root `sr_mfe.py` / `infer.py` (the reference's scripts' flags plus the B200 path's)."""
    import argparse
    ap = argparse.ArgumentParser(prog=prog)
    ap.add_argument('-c', '--config', type=str, default=default_config, help='JSON file for configuration')
    ap.add_argument('-p', '--phase', type=str, choices=['train', 'val'], default='val')
    ap.add_argument('-gpu', '--gpu_ids', type=str, default=None)
    ap.add_argument('-debug', '-d', action='store_true')
    ap.add_argument('-enable_wandb', action='store_true')
    ap.add_argument('-log_wandb_ckpt', action='store_true')
    ap.add_argument('-log_eval', action='store_true')
    ap.add_argument('-log_infer', action='store_true')
    ap.add_argument('--batch', type=int, default=16, help='images per GPU per sampling call (reference: 1)')
    ap.add_argument('--no-save', action='store_true', help='do not write SR images')
    ap.add_argument('--max-images', type=int, default=None)
    ap.add_argument('--dtype', default=os.environ.get("FDSR_DTYPE", "auto"), choices=["auto", "fp16", "bf16", "fp32"])
    ap.add_argument('--tile', type=int, default=None,
                    help='sample each image as overlapping tiles of this size (multiple of 8): scenes of any size, one per call')
    ap.add_argument('--tile-overlap', type=int, default=32, help='overlap of neighbouring tiles in pixels (with --tile)')
    ap.add_argument('--tile-batch', type=int, default=16, help='tiles per UNet call (with --tile)')
    ap.add_argument('--tile-split', action='store_true',
                    help='under torchrun, split the tiles of each image over the ranks instead of sharding the images '
                         '(with --tile): one large scene on every GPU, the single-GPU result')
    ap.add_argument('--max-value', type=int, default=None, metavar='N',
                    help='16-bit data with white level N (1..65535, e.g. 4095 for 12-bit, 65535 for 16-bit): sets '
                         'datasets.val.max_value')
    ap.add_argument('--nodata', type=int, default=None, metavar='V',
                    help='fill value of the scenes (0..255, or 0..65535 for 16-bit data): pixels whose bands all equal '
                         'V are not scored, are written as V and, with --tile, skip the UNet; sets datasets.val.nodata')
    args = ap.parse_args(argv)
    if args.tile_split and args.tile is None:
        ap.error('--tile-split needs --tile')
    if args.max_value is not None and not 1 <= args.max_value <= 65535:
        ap.error('--max-value must be 1..65535')
    if args.nodata is not None:
        if not 0 <= args.nodata <= 65535:
            ap.error('--nodata must be 0..65535')
        if args.tile_split:
            ap.error('--nodata cannot be combined with --tile-split (masked tiles are sampled on one GPU)')
    return args


def load_opt(args):
    """The run's options: the JSON config (or the programmatic equivalent of a shipped one) with the flags applied."""
    from . import config as Cfg
    cfg_path = args.config
    if os.path.exists(cfg_path) or os.path.basename(cfg_path) in Cfg._ALIASES:
        opt = Cfg.load_config(cfg_path, phase='val', gpu_ids=args.gpu_ids)
    else:  # the reference tree (and its JSON files) is absent: programmatic equivalent of the shipped config
        opt = Cfg.default_config(os.path.basename(cfg_path))
    opt["model"]["compute_dtype"] = args.dtype
    if args.max_value is not None:
        opt['datasets']['val']['max_value'] = args.max_value
    if args.nodata is not None:
        opt['datasets']['val']['nodata'] = args.nodata
    return opt


def main(argv=None, default_config="config/sr_fastdiffsr_test_64_256.json", prog="sr_mfe.py"):
    """Shared driver of the repo-root `sr_mfe.py` / `infer.py` (same flags as the reference's scripts)."""
    from .networks import define_G

    args = parse_args(argv, default_config, prog)
    if args.phase == 'train':
        raise NotImplementedError("training is outside the B200 sampling path: train with the reference and point "
                                  "path.resume_state at the checkpoint")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    opt = load_opt(args)
    paths = opt['path'] or {}
    logger = setup_logger("base", paths.get('log') if isinstance(paths, dict) else None)
    dev = torch.device("cuda", local_rank)
    netG = define_G(opt).to(dev)
    # the reference's order (model/model.py:19-41, sr_mfe.py:93-94): loss, 'train' schedule (registers the 12 buffers a
    # checkpoint carries), strict checkpoint load, then the 'val' schedule
    netG.set_loss(dev)
    netG.set_new_noise_schedule(opt['model']['beta_schedule']['train'], dev)
    if not load_network(netG, opt, logger):
        logger.warning("no path.resume_state in the config: sampling with RANDOM-INIT weights")
    netG.set_new_noise_schedule(opt['model']['beta_schedule']['val'], dev)
    netG.eval()
    if args.tile_split and dist.is_initialized():
        # the ranks evaluate different tiles of one image: they must run the same network (a random init differs per rank)
        for t in netG.state_dict().values():
            dist.broadcast(t, src=0)
        netG.refresh_weights()
    val_opt = opt['datasets']['val']
    from .data import create_dataset
    val_set = create_dataset(val_opt, 'val', channels=int(opt['model']['unet']['out_channel']))
    logger.info('Dataset [{:s} - {:s}] is created: {} images.'.format("LRHRDataset", str(val_opt['name']), len(val_set)))
    scale = int(val_opt['r_resolution']) // int(val_opt['l_resolution'])
    result_path = None if args.no_save else (paths.get('results') if isinstance(paths, dict) and paths.get('results') else 'results')
    res = evaluate(netG, val_set, batch_size=args.batch, scale=scale, result_path=result_path,
                   save_ext="png" if prog == "infer.py" else "tif", logger=logger, max_images=args.max_images,
                   tile=args.tile, tile_overlap=args.tile_overlap, tile_batch=args.tile_batch, tile_split=args.tile_split)
    if dist.is_initialized():
        dist.destroy_process_group()
    return res
