"""Test-set loaders for the entry points (the reference's utils/utils_datasets.py:61-136 on the
inference path). Disk I/O is outside the accelerated path (SURVEY 2 #12): this module only has to
yield the same 5-tuples `(Lr_SAI_y[1,1,AH,AW], Hr_SAI_y, Sr_SAI_cbcr, [angRes_in, angRes_out], [name])`
the reference's DataLoader(batch_size=1) yields. h5 datasets need h5py; `--synthetic N` produces
seeded scenes so the whole entry point can run without any dataset."""
import os

import numpy as np
import torch


def _batch1(lr, hr, cbcr, ang_in, ang_out, name):
    return (lr[None], hr[None], cbcr[None], [torch.tensor([ang_in]), torch.tensor([ang_out])], [name])


class SyntheticTestSet:
    def __init__(self, args, n, size):
        self.args, self.n, self.size = args, n, size

    def __len__(self):
        return self.n

    def __getitem__(self, i):
        if not 0 <= i < self.n:
            raise IndexError(i)
        A, s, h = self.args.angRes_in, self.args.scale_factor, self.size
        rs = np.random.RandomState(1000 + i)
        lr = torch.from_numpy(rs.random_sample((1, A * h, A * h)).astype(np.float32))
        hr = torch.from_numpy(rs.random_sample((1, A * h * s, A * h * s)).astype(np.float32))
        cbcr = torch.full((2, A * h * s, A * h * s), 0.5)
        return _batch1(lr, hr, cbcr, A, self.args.angRes_out, "synthetic_%02d" % i)

    def __iter__(self):
        for i in range(self.n):
            yield self[i]


class H5TestSet:
    """one dataset directory <path_for_test>/SR_AxA_sx/<data_name>/*.h5 (utils_datasets.py:87-136)."""

    def __init__(self, args, data_name):
        try:
            import h5py  # noqa: F401
        except ImportError as e:
            raise RuntimeError("reading .h5 test sets needs h5py, which is not installed; use --synthetic N") from e
        self.args = args
        self.root = os.path.join(args.path_for_test, "SR_%dx%d_%dx" % (args.angRes_in, args.angRes_in, args.scale_factor),
                                 data_name)
        self.files = sorted(os.listdir(self.root))

    def __len__(self):
        return len(self.files)

    def __getitem__(self, i):
        """reads only the i-th file (a rank of a multi-GPU run opens just the scenes it runs)"""
        import h5py
        fn = self.files[i]
        with h5py.File(os.path.join(self.root, fn), "r") as hf:
            lr = np.array(hf.get("Lr_SAI_y")).T
            hr = np.array(hf.get("Hr_SAI_y")).T
            cb = np.array(hf.get("Sr_SAI_cbcr"), dtype="single")
        if cb.ndim == 3:
            cb = np.transpose(cb, (2, 1, 0))
        elif cb.ndim == 0 or cb.size == 0:
            cb = np.zeros((hr.shape[0], hr.shape[1], 2), np.float32)
        elif cb.ndim == 2:
            cb = cb[..., None]
        to_t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32))
        return _batch1(to_t(lr)[None], to_t(hr)[None], to_t(cb).permute(2, 0, 1).contiguous(), self.args.angRes_in,
                       self.args.angRes_out, fn.split(".")[0])

    def __iter__(self):
        for i in range(len(self.files)):
            yield self[i]


def MultiTestSetDataLoader(args):
    if getattr(args, "synthetic", 0) > 0:
        ds = SyntheticTestSet(args, args.synthetic, args.synthetic_size)
        return ["Synthetic"], [ds], len(ds)
    base = os.path.join(args.path_for_test, "SR_%dx%d_%dx" % (args.angRes_in, args.angRes_in, args.scale_factor))
    names = sorted(os.listdir(base)) if args.data_name == "ALL" else [args.data_name]
    loaders = [H5TestSet(args, n) for n in names]
    return names, loaders, sum(len(d) for d in loaders)
