"""VTAB-1k data access for the entry point (reference image_classification/vtab.py).

Only the pieces the hot path's CLI needs survive (SURVEY section 2, row 4): the dataset names with their
class counts (reference vtab.py:9-34) and ``get_data``.  When ``./data/vtab-1k/<name>`` is absent -- as on
the benchmark boxes, which have no datasets -- ``get_data`` returns synthetic loaders with the reference's
shapes (x ~ N(0,1) [B,3,224,224] as after Normalize, labels uniform over the classes; train batch 64 with
drop_last over 1000 images, val batch 256).  The real-file path (PIL decode, bicubic 224, ImageNet
normalise) follows the reference; with ``gpu_preprocess=True`` the workers only decode (uint8 HWC) and
``cara_b200.preprocess.GpuPreprocessor`` does the bit-identical resize + ToTensor + Normalize on the GPU
(``to_device(batch)`` turns either kind of batch into the model's input).
"""
import os

import torch

_CLASSES = {"cifar": 100, "caltech101": 102, "dtd": 47, "oxford_flowers102": 102, "oxford_iiit_pet": 37,
            "svhn": 10, "sun397": 397, "patch_camelyon": 2, "eurosat": 10, "resisc45": 45,
            "diabetic_retinopathy": 5, "clevr_count": 8, "clevr_dist": 6, "dmlab": 6, "kitti": 4,
            "dsprites_loc": 16, "dsprites_ori": 16, "smallnorb_azi": 18, "smallnorb_ele": 9}
_DATASET_NAME = tuple(_CLASSES)


def get_classes_num(dataset_name):
    return _CLASSES[dataset_name]


class SyntheticImages(torch.utils.data.Dataset):
    """Deterministic N(0,1) images / uniform labels of the VTAB-1k shape."""

    def __init__(self, length, num_classes, seed, img=224):
        g = torch.Generator().manual_seed(seed)
        self.x = torch.randn(length, 3, img, img, generator=g)
        self.y = torch.randint(0, num_classes, (length,), generator=g)

    def __len__(self):
        return self.x.shape[0]

    def __getitem__(self, i):
        return self.x[i], self.y[i]


class _FileList(torch.utils.data.Dataset):
    def __init__(self, root, flist, decode_only=False, img_size=224):
        from torchvision import transforms
        self.root = root
        self.decode_only = decode_only
        with open(flist) as f:
            self.items = [(p, int(lab)) for p, lab in (ln.split() for ln in f if ln.strip())]
        self.tf = transforms.Compose([
            transforms.Resize((img_size, img_size), interpolation=transforms.InterpolationMode.BICUBIC),
            transforms.ToTensor(),
            transforms.Normalize(mean=[0.485, 0.456, 0.406], std=[0.229, 0.224, 0.225])])

    def __len__(self):
        return len(self.items)

    def __getitem__(self, i):
        from PIL import Image
        path, lab = self.items[i]
        img = Image.open(os.path.join(self.root, path)).convert("RGB")
        if self.decode_only:
            import numpy as np
            return np.asarray(img), lab
        return self.tf(img), lab


def _collate_decoded(batch):
    """Decoded images keep their own sizes: a list of uint8 [H,W,3] arrays + the label tensor."""
    return [b[0] for b in batch], torch.as_tensor([b[1] for b in batch])


_PRE = {}


def to_device(x, y, device="cuda", size=224):
    """A loader batch -> (fp32 [B,3,size,size], labels) on the device; decoded uint8 batches go through the GPU
    resize / normalise kernels."""
    if isinstance(x, (list, tuple)):
        from cara_b200.preprocess import GpuPreprocessor
        dev = torch.device(device)
        if dev.index is None and dev.type == "cuda":
            dev = torch.device("cuda", torch.cuda.current_device())
        pre = _PRE.get((dev, size))
        if pre is None:
            pre = _PRE[(dev, size)] = GpuPreprocessor(dev, size=size)
        return pre(x), y.to(dev, non_blocking=True)
    return x.to(device, non_blocking=True), y.to(device, non_blocking=True)


def get_data(name, evaluate=True, batch_size=64, synthetic=None, train_len=1000, val_len=512, gpu_preprocess=False,
             img_size=224):
    root = "./data/vtab-1k/" + name
    if synthetic is None:
        synthetic = not os.path.isdir(root)
    if synthetic:
        print(f"Synthetic VTAB-1k-shaped data for {name} ({root} not used)")
        k = get_classes_num(name)
        train, val = SyntheticImages(train_len, k, 1, img=img_size), SyntheticImages(val_len, k, 2, img=img_size)
        workers = 0
    else:
        print(f"Getting data from root: {root}")
        tr, va = ("/train800val200.txt", "/test.txt") if evaluate else ("/train800.txt", "/val200.txt")
        train = _FileList(root, root + tr, gpu_preprocess, img_size)
        val = _FileList(root, root + va, gpu_preprocess, img_size)
        workers = 4
    collate = _collate_decoded if (gpu_preprocess and not synthetic) else None
    train_loader = torch.utils.data.DataLoader(train, batch_size=batch_size, shuffle=True, drop_last=True,
                                               num_workers=workers, pin_memory=collate is None, collate_fn=collate)
    val_loader = torch.utils.data.DataLoader(val, batch_size=256, shuffle=False, num_workers=workers,
                                             pin_memory=collate is None, collate_fn=collate)
    return train_loader, val_loader
