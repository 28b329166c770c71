"""Validation data path: the reference's folder-of-images LR/HR dataset (data/LRHR_dataset.py:10-128,
datatype 'img'; data/util.py:9-24 file discovery) with a batched, prefetching loader.

The reference's val loader yields one image per step from one worker (data/__init__.py:16-18) and
reads a *precomputed* bicubic image from `sr_{l}_{r}/`.  At thousands of images per second that
loader is the bottleneck (SURVEY 8f N2), so here
  * items are decoded to uint8 (the reference's ToTensor + *2-1 happens on the device, bit-identically);
  * `sr_{l}_{r}/` is optional: the library's bit-exact PIL bicubic (`fdsr_bicubic_u8`) rebuilds it from
    `lr_{l}/` (SURVEY F3), and when the folder exists it is used as is, like the reference does;
  * batches are assembled in pinned memory by a background thread one batch ahead of the GPU;
  * images of C = 1..8 bands (`channels`, the UNet's out_channel): C = 3 reads RGB images exactly as the reference,
    C = 1 reads images as single-band 'L' or `.npy` arrays, any other C reads `.npy` (H,W,C) uint8 arrays;
  * 16-bit imagery (`max_value` = M, the white level that maps to +1, DESIGN.md §4.6): `.npy` (H,W,C) uint16 arrays
    for any C, and for C = 1 also 16-bit single-band images (Pillow modes I;16 / I;16L / I;16B, or I with values in
    0..65535); items stay uint16 up to the device, where `u16_to_tensor` normalises them with M.
"""
from __future__ import annotations

import os
import queue
import threading

import numpy as np
import torch

IMG_EXTENSIONS = ['.jpg', '.JPG', '.jpeg', '.JPEG', '.png', '.PNG', '.ppm', '.PPM', '.bmp', '.BMP', 'tif']


def is_image_file(filename):
    return any(filename.endswith(ext) for ext in IMG_EXTENSIONS)


def _is_band_file(filename, channels, wide=False):
    """Files an image folder of `channels` bands is made of: images for C = 3, images or .npy for C = 1, .npy else.
    A 16-bit folder (`wide`) is made of .npy and image files for every C; the loader rejects what it cannot read."""
    if wide:
        return filename.endswith(".npy") or is_image_file(filename)
    if channels == 3:
        return is_image_file(filename)
    return filename.endswith(".npy") or (channels == 1 and is_image_file(filename))


def get_paths_from_images(path, channels=3, wide=False):
    """data/util.py:13-24 (channels=3); other band counts and 16-bit folders (`wide`) keep the files _is_band_file
    accepts."""
    assert os.path.isdir(path), '{:s} is not a valid directory'.format(path)
    images, rejected = [], 0
    for dirpath, _, fnames in sorted(os.walk(path)):
        for fname in sorted(fnames):
            if _is_band_file(fname, channels, wide):
                images.append(os.path.join(dirpath, fname))
            elif is_image_file(fname):
                rejected += 1
    if not images and rejected:
        raise ValueError(f"{path}: {channels}-band images must be .npy (H,W,{channels}) uint8 arrays; the folder holds "
                         f"{rejected} image file(s), which are read only for 1 or 3 bands")
    assert images, '{:s} has no valid image file'.format(path)
    return sorted(images)


def _pil_u8(im, channels):
    """A PIL image as (H,W,C) uint8: RGB for C = 3, one 'L' band for C = 1 (copy: PIL buffers are read-only)."""
    if channels == 3:
        return np.array(im.convert("RGB"), dtype=np.uint8)
    return np.array(im.convert("L"), dtype=np.uint8)[:, :, None]


def _load_u8(path, channels=3):
    if path.endswith(".npy"):
        a = np.load(path, allow_pickle=False)
        if a.ndim == 2 and channels == 1:
            a = a[:, :, None]
        if a.dtype != np.uint8 or a.ndim != 3 or a.shape[2] != channels:
            raise ValueError(f"{path}: expected a (H,W,{channels}) uint8 array, got {a.dtype} {a.shape}")
        return np.ascontiguousarray(a)
    from PIL import Image
    with Image.open(path) as im:
        return _pil_u8(im, channels)


_I16_MODES = ("I;16", "I;16L", "I;16B")


def _load_u16(path, channels):
    """A file of a 16-bit dataset as (H,W,C) uint16: a .npy uint16 array ((H,W) too for C = 1), or for C = 1 a 16-bit
    single-band image (I;16 / I;16L / I;16B, or I with values in 0..65535), read losslessly.  Anything else is a
    ValueError naming the file."""
    if path.endswith(".npy"):
        a = np.load(path, allow_pickle=False)
        if a.ndim == 2 and channels == 1:
            a = a[:, :, None]
        if a.dtype != np.uint16 or a.ndim != 3 or a.shape[2] != channels:
            raise ValueError(f"{path}: a 16-bit dataset of {channels} band(s) needs (H,W,{channels}) uint16 arrays, got "
                             f"{a.dtype} {a.shape}")
        return np.ascontiguousarray(a)
    from PIL import Image
    with Image.open(path) as im:
        mode = im.mode
        if channels != 1:
            raise ValueError(f"{path}: a 16-bit dataset of {channels} bands is read from .npy (H,W,{channels}) uint16 "
                             f"arrays, not from {mode} images")
        if mode in _I16_MODES:
            a = np.asarray(im).astype(np.uint16)
        elif mode == "I":
            a = np.asarray(im)
            if a.size and (a.min() < 0 or a.max() > 65535):
                raise ValueError(f"{path}: mode I image with values outside 0..65535")
            a = a.astype(np.uint16)
        else:
            raise ValueError(f"{path}: a 16-bit single-band dataset needs I;16 (or I) images, got mode {mode}")
    return np.ascontiguousarray(a)[:, :, None]


def u16_to_tensor(img_u16: torch.Tensor, max_value: int):
    """(B,H,W,C) uint16 -> (B,C,H,W) fp32 in [-1,1] at white level M = max_value: (min(v, M) / M) * 2 - 1 in fp32,
    each step rounded to nearest (fdsr_bicubic_u16's conditioning bit for bit).  The divisor is a tensor on the
    data's device, so that no device divides by a reciprocal of M."""
    v = img_u16.permute(0, 3, 1, 2).float().clamp(max=float(max_value))
    return (v / torch.tensor(float(max_value), dtype=torch.float32, device=v.device)) * 2.0 - 1.0


def nodata_mask(img: torch.Tensor, nodata: int, H: int, W: int):
    """The (B,H,W) bool validity mask at the HR size H x W of a (B,h,w,C) uint8 / uint16 image: a source pixel is
    invalid iff every band equals `nodata`, and HR pixel (Y, X) takes source pixel (((2Y+1) h) // (2H),
    ((2X+1) w) // (2W)), the one whose area holds the HR pixel's centre (the identity at h = H, w = W).  The bicubic
    conditioning mixes fill into the valid pixels within two LR pixels of the footprint edge; that halo is scored and
    sampled as valid, not corrected."""
    if img.dim() != 4 or img.dtype not in (torch.uint8, torch.uint16):
        raise ValueError(f"nodata_mask needs a (B,h,w,C) uint8 or uint16 tensor, got {img.dtype} {tuple(img.shape)}")
    _, h, w, _ = img.shape
    valid = (img != nodata).any(dim=3)
    ys = (torch.arange(H, device=img.device) * 2 + 1) * h // (2 * H)
    xs = (torch.arange(W, device=img.device) * 2 + 1) * w // (2 * W)
    return valid[:, ys][:, :, xs]


def u8_to_tensor(img_u8: torch.Tensor):
    """(B,H,W,C) uint8 -> (B,C,H,W) fp32 in [-1,1]: torchvision ToTensor (/255) then *2-1
    (data/util.py:66-75 with min_max=(-1,1)), same operation order."""
    return (img_u8.permute(0, 3, 1, 2).float() / 255.0) * 2.0 - 1.0


def _decode_u8(buf, channels=3):
    from io import BytesIO
    from PIL import Image
    with Image.open(BytesIO(buf)) as im:
        return _pil_u8(im, channels)


class _LmdbStore:
    """Read-only view of an LMDB environment written by the reference's data/prepare_data_mfe_dm.py (keys
    `hr_{r}_{idx:05d}`, `sr_{l}_{r}_{idx:05d}`, `lr_{l}_{idx:05d}`, `length`), opened exactly as
    data/LRHR_dataset.py:17-19 does.  Needs the `lmdb` package, like the reference."""

    def __init__(self, dataroot):
        try:
            import lmdb
        except ImportError as e:
            raise ImportError("datatype 'lmdb' needs the `lmdb` package (the reference imports it too, "
                              "data/LRHR_dataset.py:2); install it or export the dataset to image folders") from e
        self.env = lmdb.open(dataroot, readonly=True, lock=False, readahead=False, meminit=False)

    def get(self, key: bytes):
        with self.env.begin(write=False) as txn:
            v = txn.get(key)
            return None if v is None else bytes(v)


class LRHRDataset:
    """The reference's validation dataset (data/LRHR_dataset.py:9-128): datatype 'img' = folder layout
    `{dataroot}/hr_{r}`, `{dataroot}/lr_{l}`, optional `{dataroot}/sr_{l}_{r}`; datatype 'lmdb' = the key-value layout
    of data/LRHR_dataset.py:17-27, 60-93 (`kv`: any object with get(key: bytes) -> bytes | None; default: the LMDB
    environment at `dataroot`).  `channels`: bands per image (1..8, see the module docstring); 'lmdb' holds
    encoded images and so serves 1 or 3 bands.  `max_value`: None = 8-bit data; an integer M in 1..65535 = 16-bit
    data with white level M (datatype 'img' only), read by `_load_u16` and normalised by `u16_to_tensor`.
    `nodata`: None, or the sample value V that marks fill (0..255 for 8-bit data, 0..65535 with max_value): a pixel
    whose bands all equal V is outside the scene's footprint (nodata_mask)."""

    def __init__(self, dataroot, datatype="img", l_resolution=64, r_resolution=256, split="val", data_len=-1,
                 need_LR=True, img_mask="no", kv=None, channels=3, max_value=None, nodata=None):
        if datatype not in ("img", "lmdb"):
            raise NotImplementedError('data_type [{:s}] is not recognized.'.format(str(datatype)))
        if max_value is not None:
            if isinstance(max_value, bool) or int(max_value) != max_value or not 1 <= int(max_value) <= 65535:
                raise ValueError(f"max_value must be an integer 1..65535 (got {max_value!r})")
            max_value = int(max_value)
            if datatype != "img":
                raise ValueError(f"max_value: 16-bit data is read from image folders (datatype 'img'); datatype "
                                 f"'{datatype}' stores encoded 8-bit images")
        self.max_value = max_value
        if nodata is not None:
            top = 255 if max_value is None else 65535
            if isinstance(nodata, bool) or int(nodata) != nodata or not 0 <= int(nodata) <= top:
                raise ValueError(f"nodata must be an integer 0..{top} for {'8' if max_value is None else '16'}-bit data "
                                 f"(got {nodata!r})")
            nodata = int(nodata)
        self.nodata = nodata
        if not 1 <= int(channels) <= 8:
            raise ValueError(f"channels must be 1..8 (got {channels})")
        if datatype == "lmdb" and channels not in (1, 3):
            raise ValueError(f"datatype 'lmdb' stores encoded images and serves 1 or 3 bands, not {channels}: export the "
                             "dataset to folders of .npy (H,W,C) uint8 arrays")
        self.channels = int(channels)
        if split == "train":
            raise NotImplementedError("the training data path (random flips) is outside the B200 sampling path")
        self.l_res, self.r_res, self.split = l_resolution, r_resolution, split
        self.datatype = datatype
        self.need_LR = need_LR
        if datatype == "lmdb":
            self.kv = kv if kv is not None else _LmdbStore(dataroot)
            length = self.kv.get("length".encode("utf-8"))
            if length is None:
                raise ValueError(f"{dataroot}: no 'length' key — not a dataset written by prepare_data_mfe_dm.py")
            self.dataset_len = int(length)
            self.data_len = self.dataset_len if (data_len is None or data_len <= 0) else min(data_len, self.dataset_len)
            return
        wide = max_value is not None
        self.hr_path = get_paths_from_images('{}/hr_{}'.format(dataroot, r_resolution), self.channels, wide)
        sr_dir = '{}/sr_{}_{}'.format(dataroot, l_resolution, r_resolution)
        lr_dir = '{}/lr_{}'.format(dataroot, l_resolution)
        self.sr_path = get_paths_from_images(sr_dir, self.channels, wide) if os.path.isdir(sr_dir) else None
        self.lr_path = get_paths_from_images(lr_dir, self.channels, wide) if os.path.isdir(lr_dir) else None
        if self.sr_path is None and self.lr_path is None:
            raise FileNotFoundError(f"{dataroot}: neither {os.path.basename(sr_dir)}/ nor {os.path.basename(lr_dir)}/ exists")
        for p in (self.sr_path, self.lr_path):
            if p is not None and len(p) != len(self.hr_path):
                raise ValueError(f"{dataroot}: folder sizes differ ({len(p)} vs {len(self.hr_path)} HR images)")
        self.dataset_len = len(self.hr_path)
        self.data_len = self.dataset_len if (data_len is None or data_len <= 0) else min(data_len, self.dataset_len)

    def __len__(self):
        return self.data_len

    def _lmdb_u8(self, index):
        tag = str(index).zfill(5)
        keys = {"HR": 'hr_{}_{}'.format(self.r_res, tag), "SR": 'sr_{}_{}_{}'.format(self.l_res, self.r_res, tag),
                "LR": 'lr_{}_{}'.format(self.l_res, tag)}
        raw = {k: self.kv.get(v.encode("utf-8")) for k, v in keys.items() if k != "LR" or self.need_LR}
        # The reference replaces an invalid index by a RANDOM valid one (data/LRHR_dataset.py:77-92), which silently
        # evaluates some image twice; validation here must be reproducible, so a hole in the store is an error
        if raw["HR"] is None or (raw["SR"] is None and raw.get("LR") is None):
            raise KeyError(f"lmdb dataset: index {index} has no {keys['HR']} / {keys['SR']} entry")
        item = {k: _decode_u8(v, self.channels) for k, v in raw.items() if v is not None}
        item["Index"] = index
        item["path"] = keys["HR"]
        return item

    def get_raw(self, index):
        """HWC arrays as stored, uint8 (8-bit data) or uint16 (max_value set): always 'HR'; 'LR' and/or 'SR' as present
        on disk."""
        if self.datatype == "lmdb":
            return self._lmdb_u8(index)
        load = _load_u8 if self.max_value is None else _load_u16
        item = {"HR": load(self.hr_path[index], self.channels), "Index": index, "path": self.hr_path[index]}
        if self.lr_path is not None:
            item["LR"] = load(self.lr_path[index], self.channels)
        if self.sr_path is not None:
            item["SR"] = load(self.sr_path[index], self.channels)
        return item

    def get_u8(self, index):
        """uint8 HWC arrays of an 8-bit dataset (get_raw); a 16-bit dataset has no uint8 form."""
        if self.max_value is not None:
            raise ValueError("a 16-bit dataset (max_value set) holds uint16 arrays: use get_raw")
        return self.get_raw(index)

    def to_tensor(self, img):
        """(B,H,W,C) stored arrays -> (B,C,H,W) fp32 in [-1,1]: u8_to_tensor, or u16_to_tensor at max_value."""
        return u8_to_tensor(img) if self.max_value is None else u16_to_tensor(img, self.max_value)

    def __getitem__(self, index):
        """The reference's item (fp32 CHW tensors in [-1,1]; 'SR' needs the sr_ folder)."""
        it = self.get_raw(index)
        out = {"Index": index}
        for k in ("HR", "SR", "LR"):
            if k in it:
                out[k] = self.to_tensor(torch.from_numpy(it[k])[None])[0]
        return out


def create_dataset(dataset_opt, phase, channels=3):
    """data/__init__.py:24-40; `channels`: bands per image (the UNet's out_channel); `dataset_opt['max_value']`: the
    white level of 16-bit data (absent or None: 8-bit data); `dataset_opt['nodata']`: the fill value (absent or None:
    every pixel is valid)."""
    return LRHRDataset(dataroot=dataset_opt['dataroot'], datatype=dataset_opt['datatype'],
                       l_resolution=dataset_opt['l_resolution'], r_resolution=dataset_opt['r_resolution'],
                       split=phase, data_len=dataset_opt['data_len'] if dataset_opt['data_len'] is not None else -1,
                       need_LR=(dataset_opt['mode'] == 'LRHR'), channels=channels,
                       max_value=dataset_opt.get('max_value'), nodata=dataset_opt.get('nodata'))


class BatchLoader:
    """Iterates `indices` of a dataset in batches of its stored arrays (uint8, or uint16 for 16-bit data) stacked in
    pinned host memory, decoding one batch ahead in a background thread.  Yields dicts
    {'HR','LR'?,'SR'?: pinned (B,H,W,C), 'Index': list}."""

    def __init__(self, dataset, batch_size, indices=None, prefetch=2, pin=True):
        self.ds = dataset
        self.bs = max(1, int(batch_size))
        self.indices = list(range(len(dataset))) if indices is None else list(indices)
        self.prefetch = prefetch
        self.pin = pin and torch.cuda.is_available()

    def __len__(self):
        return (len(self.indices) + self.bs - 1) // self.bs

    def _assemble(self, idxs):
        items = [self.ds.get_raw(i) for i in idxs]
        out = {"Index": list(idxs), "path": [it["path"] for it in items]}
        for k in ("HR", "LR", "SR"):
            if k in items[0]:
                arr = torch.from_numpy(np.stack([it[k] for it in items], 0))
                out[k] = arr.pin_memory() if self.pin else arr
        return out

    def __iter__(self):
        q = queue.Queue(maxsize=self.prefetch)
        chunks = [self.indices[i:i + self.bs] for i in range(0, len(self.indices), self.bs)]

        def work():
            try:
                for ch in chunks:
                    q.put(self._assemble(ch))
                q.put(None)
            except BaseException as e:  # surface decode errors in the consumer
                q.put(e)

        th = threading.Thread(target=work, daemon=True)
        th.start()
        while True:
            item = q.get()
            if item is None:
                break
            if isinstance(item, BaseException):
                raise item
            yield item
