"""Minimal rectangular validation loader: the harness that feeds `DetectionValidator` the batches the reference's
`YOLODataset(rect=True, augment=False)` + `build_dataloader(shuffle=False)` would produce (reference
data/dataset.py:137-165 load_image, :211-235 set_rectangle, :274-290 transforms, :325-342 collate_fn;
data/augment.py:636-700 LetterBox(scaleup=False) + label update, :929-956 Format).

Scope: labelled image folders in YOLO txt format, rect batches, no augmentation, no caching, no workers: enough to run
`YOLOLite.val(data=...)` on a coco8-style dataset.  Training-side dataset features (mosaic, mixup, caches, segment /
keypoint labels) are out of scope.  Image decode/resize is cv2 on the host exactly like the reference, so the batch is
bit-identical to the reference's (pinned by tests/golden/real_images.npz)."""
from __future__ import annotations

import math
from pathlib import Path

import numpy as np
import torch

from .augment import LetterBox

IMG_FORMATS = {"bmp", "jpeg", "jpg", "png", "tif", "tiff", "webp"}


def read_yolo_labels(path) -> np.ndarray:
    """(n, 5) float32 [cls, x, y, w, h] normalised, duplicates removed like the reference (data/utils.py:73-91)."""
    p = Path(path)
    if not p.is_file():
        return np.zeros((0, 5), np.float32)
    rows = [x.split() for x in p.read_text().strip().splitlines() if len(x)]
    lb = np.array(rows, dtype=np.float32).reshape(-1, 5) if rows else np.zeros((0, 5), np.float32)
    if len(lb):
        _, i = np.unique(lb, axis=0, return_index=True)
        if len(i) < len(lb):
            lb = lb[i]
    return lb[:, :5]


class RectValLoader:
    """Iterable of batch dicts (`img` uint8 BCHW RGB, `cls`, `bboxes` normalised xywh, `batch_idx`, `ori_shape`,
    `resized_shape`, `ratio_pad`, `im_file`) over `images`, in the reference's rect order (ascending h/w)."""

    def __init__(self, images, labels, imgsz=640, batch_size=16, stride=32, pad=0.5, im_files=None):
        """`images`: list of BGR uint8 HWC arrays or file paths; `labels`: list of (n, 5) [cls, xywh-normalised]."""
        import cv2

        self.imgsz, self.batch_size, self.stride, self.pad = int(imgsz), int(batch_size), int(stride), float(pad)
        ims = []
        for im in images:
            if not isinstance(im, np.ndarray):
                arr = cv2.imread(str(im))
                if arr is None:
                    raise FileNotFoundError(f"cannot read image {im}")
                im = arr
            ims.append(im)
        files = list(im_files) if im_files is not None else [str(i) if isinstance(i, (str, Path)) else f"image{k}"
                                                            for k, i in enumerate(images)]
        labels = [np.asarray(lb, np.float32).reshape(-1, 5) for lb in labels]
        assert len(ims) == len(labels) == len(files)
        # set_rectangle (dataset.py:211-235): sort by aspect ratio h/w, one shape per batch
        ni = len(ims)
        bi = np.floor(np.arange(ni) / self.batch_size).astype(int)
        nb = int(bi[-1]) + 1 if ni else 0
        s = np.array([im.shape[:2] for im in ims], dtype=np.float64).reshape(-1, 2)
        ar = s[:, 0] / s[:, 1]
        irect = ar.argsort()
        self.ims = [ims[i] for i in irect]
        self.labels = [labels[i] for i in irect]
        self.im_files = [files[i] for i in irect]
        ar = ar[irect]
        shapes = [[1, 1]] * nb
        for i in range(nb):
            ari = ar[bi == i]
            mini, maxi = ari.min(), ari.max()
            if maxi < 1:
                shapes[i] = [maxi, 1]
            elif mini > 1:
                shapes[i] = [1, 1 / mini]
        self.batch_shapes = (np.ceil(np.array(shapes) * self.imgsz / self.stride + self.pad).astype(int) * self.stride
                             if nb else np.zeros((0, 2), int))
        self.batch = bi

    @classmethod
    def from_dirs(cls, img_dir, label_dir=None, **kw):
        img_dir = Path(img_dir)
        files = sorted(str(p) for p in img_dir.rglob("*.*") if p.suffix[1:].lower() in IMG_FORMATS)
        if not files:
            raise FileNotFoundError(f"no images under {img_dir}")
        return cls.from_files(files, label_dir, **kw)

    @classmethod
    def from_files(cls, files, label_dir=None, **kw):
        if label_dir is None:   # reference img2label_paths: .../images/... -> .../labels/...
            lab = [Path(f.replace("/images/", "/labels/", 1)).with_suffix(".txt") for f in files]
        else:
            lab = [Path(label_dir) / (Path(f).stem + ".txt") for f in files]
        return cls(files, [read_yolo_labels(p) for p in lab], im_files=files, **kw)

    def __len__(self):
        return int(self.batch[-1]) + 1 if len(self.ims) else 0

    def _item(self, i):
        import cv2

        im = self.ims[i]
        h0, w0 = im.shape[:2]
        r = self.imgsz / max(h0, w0)                       # load_image(rect_mode=True), dataset.py:147-151
        if r != 1:
            w, h = min(math.ceil(w0 * r), self.imgsz), min(math.ceil(h0 * r), self.imgsz)
            im = cv2.resize(im, (w, h), interpolation=cv2.INTER_LINEAR)
        rh, rw = im.shape[:2]
        new_shape = tuple(int(v) for v in self.batch_shapes[self.batch[i]])
        # LetterBox(scaleup=False, center=True) geometry (augment.py:646-668) for the label update
        rr = min(min(new_shape[0] / rh, new_shape[1] / rw), 1.0)
        new_unpad = int(round(rw * rr)), int(round(rh * rr))
        dw, dh = (new_shape[1] - new_unpad[0]) / 2, (new_shape[0] - new_unpad[1]) / 2
        top, left = int(round(dh - 0.1)), int(round(dw - 0.1))
        img = LetterBox(new_shape=new_shape, scaleup=False)(image=im)
        lb = self.labels[i]
        cls_, box = lb[:, 0:1].copy(), lb[:, 1:5].copy()
        if len(box):                                       # _update_labels: xywh(n) -> xyxy px -> scale -> pad
            xy, wh = box[:, :2].copy(), box[:, 2:] / 2
            box = np.concatenate([xy - wh, xy + wh], 1).astype(np.float32)
            for c, sc in enumerate((rw, rh, rw, rh)):
                box[:, c] *= sc
            for c in range(4):
                box[:, c] *= rr
            for c, off in enumerate((dw, dh, dw, dh)):
                box[:, c] += off
            # Format(bbox_format="xywh", normalize=True): xyxy -> xywh, divide by the letterboxed w, h
            out = np.empty_like(box)
            out[:, 0] = (box[:, 0] + box[:, 2]) / 2
            out[:, 1] = (box[:, 1] + box[:, 3]) / 2
            out[:, 2] = box[:, 2] - box[:, 0]
            out[:, 3] = box[:, 3] - box[:, 1]
            bb = torch.from_numpy(out)
            bb[:, [0, 2]] /= img.shape[1]
            bb[:, [1, 3]] /= img.shape[0]
        else:
            bb = torch.zeros((0, 4))
        chw = np.ascontiguousarray(img.transpose(2, 0, 1)[::-1])   # HWC BGR -> CHW RGB
        return {"im_file": self.im_files[i], "ori_shape": (h0, w0), "resized_shape": new_shape,
                "ratio_pad": ((rh / h0, rw / w0), (left, top)), "img": torch.from_numpy(chw),
                "cls": torch.from_numpy(cls_) if len(box) else torch.zeros(0), "bboxes": bb, "n": len(lb)}

    def __iter__(self):
        for b in range(len(self)):
            items = [self._item(i) for i in np.nonzero(self.batch == b)[0]]
            yield {
                "im_file": tuple(it["im_file"] for it in items),
                "ori_shape": tuple(it["ori_shape"] for it in items),
                "resized_shape": tuple(it["resized_shape"] for it in items),
                "ratio_pad": tuple(it["ratio_pad"] for it in items),
                "img": torch.stack([it["img"] for it in items], 0),
                "cls": torch.cat([it["cls"].view(-1, 1) for it in items], 0),
                "bboxes": torch.cat([it["bboxes"] for it in items], 0),
                "batch_idx": torch.cat([torch.full((it["n"],), float(k)) for k, it in enumerate(items)], 0),
            }


def load_data_yaml(data) -> dict:
    """A dataset yaml (keys path / val / names like coco8.yaml) with `path` resolved against the yaml's directory."""
    from ..utils import yaml_load

    p = Path(str(data))
    d = yaml_load(p)
    root = Path(d.get("path") or p.parent)
    d["path"] = root if root.is_absolute() else (p.parent / root).resolve()
    return d


def build_val_loader(data, imgsz=640, batch_size=16, stride=32, split="val"):
    """`data`: a dataset yaml (keys path / val / names like coco8.yaml; `path` must resolve) or an image directory.  The
    split is an image directory or, as in coco.yaml (`val: val2017.txt`), a `.txt` list of image paths relative to
    `path`; labels are found by the `/images/` -> `/labels/` rule either way."""
    p = Path(str(data))
    kw = dict(imgsz=imgsz, batch_size=batch_size, stride=stride)
    if p.suffix in {".yaml", ".yml"}:
        d = load_data_yaml(p)
        split_path, names = d["path"] / d[split], d.get("names")
        if split_path.suffix == ".txt":
            lines = [x.strip() for x in split_path.read_text().splitlines() if x.strip()]
            files = sorted(str(d["path"] / x) for x in lines if x.split(".")[-1].lower() in IMG_FORMATS)
            if not files:
                raise FileNotFoundError(f"no images listed in {split_path}")
            return RectValLoader.from_files(files, **kw), names
    else:
        split_path, names = p, None
    return RectValLoader.from_dirs(split_path, **kw), names
