"""Columnar structured arrays: the input-layout contract of the kernels.

Mirrors the part of lsqfitgp's StructuredArray that the GP-fitting path relies on
(reference: src/lsqfitgp/_array.py:29-411 StructuredArray, :488-504 unstructured_to_structured,
:555-564 _nd): one array per field, every leaf field (and every element of a shaped field) is
one covariate dimension.  On the device the points are stored field-major, x[d, i], which is what
the Gram kernels read (coalesced along i).

Points may also be torch tensors, or dictionaries / StructuredArrays whose leaf fields are torch tensors (on the CPU
or the GPU, possibly requiring grad): their columns stay torch tensors, so that gradients with respect to the points
reach them (the reference differentiates through the points of `gpfactory` with jax, src/lsqfitgp/_fit.py:687-702).
"""

import numpy
import torch

__all__ = ['StructuredArray', 'unstructured_to_structured', 'asarray']


class StructuredArray:
    """Read-only columnar version of a numpy structured array.

    Parameters
    ----------
    array : numpy structured array, StructuredArray, or dict name -> array
    """

    def __init__(self, array):
        if isinstance(array, StructuredArray):
            self._fields = dict(array._fields)
            self.shape = array.shape
            self.dtype = array.dtype
            return
        if isinstance(array, dict):
            self._init_from_dict(array)
            return
        array = numpy.asarray(array)
        if array.dtype.names is None:
            raise ValueError('StructuredArray needs a structured dtype; use unstructured_to_structured')
        self._fields = {}
        for name in array.dtype.names:
            col = array[name]
            if col.dtype.names is not None:
                col = StructuredArray(col)
            self._fields[name] = col
        self.shape = array.shape
        self.dtype = array.dtype

    def _init_from_dict(self, d):
        if not d:
            raise ValueError('empty dictionary')
        arrays = {k: (v if isinstance(v, (StructuredArray, torch.Tensor)) else numpy.asarray(v)) for k, v in d.items()}
        shape = None
        for k, v in arrays.items():
            s = v.shape
            shape = s if shape is None else _common_prefix(shape, s)
        descr = []
        for k, v in arrays.items():
            sub = v.shape[len(shape):]
            dt = _numpy_dtype(v)
            descr.append((k, dt, sub) if sub else (k, dt))
        self._fields = arrays
        self.shape = shape
        self.dtype = numpy.dtype(descr)

    @classmethod
    def from_dict(cls, mapping):
        return cls(dict(mapping))

    @classmethod
    def from_dataframe(cls, df):
        """ pandas / polars DataFrame -> 1-d StructuredArray, one field per column """
        return cls({str(c): numpy.asarray(df[c]) for c in df.columns})

    @property
    def size(self):
        return int(numpy.prod(self.shape, dtype=int))

    @property
    def ndim(self):
        return len(self.shape)

    def __len__(self):
        if not self.shape:
            raise TypeError('len() of unsized object')
        return self.shape[0]

    def __getitem__(self, key):
        if isinstance(key, str):
            return self._fields[key]
        if isinstance(key, list) and key and all(isinstance(k, str) for k in key):
            return StructuredArray({k: self._fields[k] for k in key})
        new = object.__new__(StructuredArray)
        new._fields = {}
        probe = numpy.empty(self.shape, dtype=bool)[key]
        for name, col in self._fields.items():
            if isinstance(col, StructuredArray):
                new._fields[name] = col[key]
            else:
                sub = col.ndim - len(self.shape)
                idx = key if isinstance(key, tuple) else (key,)
                new._fields[name] = col[idx + (Ellipsis,)] if sub else col[key]
        new.shape = probe.shape
        new.dtype = self.dtype
        return new

    def reshape(self, *shape):
        if len(shape) == 1 and isinstance(shape[0], (tuple, list)):
            shape = tuple(shape[0])
        probe = numpy.empty(self.shape, dtype=bool).reshape(shape)
        new = object.__new__(StructuredArray)
        new._fields = {}
        for name, col in self._fields.items():
            if isinstance(col, StructuredArray):
                new._fields[name] = col.reshape(probe.shape)
            else:
                sub = col.shape[len(self.shape):]
                new._fields[name] = col.reshape(probe.shape + sub)
        new.shape = probe.shape
        new.dtype = self.dtype
        return new

    @property
    def T(self):
        if self.ndim < 2:
            return self
        raise NotImplementedError('transpose of n-d StructuredArray')

    def leaf_columns(self):
        """ list of (label, flat 1-d float array) for every covariate dimension, in dtype order """
        out = []
        n = self.size
        for name, col in self._fields.items():
            if isinstance(col, StructuredArray):
                out += [((name,) + lab if isinstance(lab, tuple) else (name, lab), c) for lab, c in col.leaf_columns()]
            else:
                flat = col.reshape(n, -1) if isinstance(col, torch.Tensor) else numpy.asarray(col).reshape(n, -1)
                if flat.shape[1] == 1 and col.ndim == len(self.shape):
                    out.append((name, flat[:, 0]))
                else:
                    out += [((name, j), flat[:, j]) for j in range(flat.shape[1])]
        return out

    def __repr__(self):
        return f'StructuredArray(shape={self.shape}, fields={list(self._fields)})'


def _numpy_dtype(v):
    """ numpy dtype of a field: a torch tensor's maps to the numpy dtype of the same name """
    if isinstance(v, torch.Tensor):
        return numpy.dtype(str(v.dtype).removeprefix('torch.'))
    return v.dtype


def _common_prefix(a, b):
    out = []
    for x, y in zip(a, b):
        if x != y:
            break
        out.append(x)
    return tuple(out)


def unstructured_to_structured(arr, dtype=None, names=None, **_):
    """ like numpy.lib.recfunctions.unstructured_to_structured: last axis -> fields """
    arr = numpy.asarray(arr)
    nf = arr.shape[-1]
    if dtype is not None:
        names = numpy.dtype(dtype).names
    if names is None:
        names = [f'f{i}' for i in range(nf)]
    if len(names) != nf:
        raise ValueError('number of names does not match the last axis')
    return StructuredArray({n: arr[..., i] for i, n in enumerate(names)})


def asarray(x):
    """ numpy array, or StructuredArray for structured inputs; a torch tensor is returned as it is """
    if isinstance(x, (StructuredArray, torch.Tensor)):
        return x
    if isinstance(x, dict):
        return StructuredArray(x)
    try:
        import pandas
        if isinstance(x, pandas.DataFrame):
            return StructuredArray.from_dataframe(x)
    except ImportError:  # pragma: no cover
        pass
    x = numpy.asarray(x)
    if x.dtype.names is not None:
        return StructuredArray(x)
    return x


_REAL_INT = (torch.bool, torch.uint8, torch.int8, torch.int16, torch.int32, torch.int64)


def _check_tensor_dtype(t):
    if not (t.dtype.is_floating_point or t.dtype in _REAL_INT):
        raise TypeError(f'points have non-real dtype {t.dtype!r}')


def columns_of(x):
    """ (labels, (ndim, n) float64 array, shape) of an array-like of points.  The array is numpy, or a torch tensor
    (on the device of the first tensor column) when the points or any of their fields are torch tensors: built with
    torch operations, it stays on the autograd graph of the points. """
    x = asarray(x)
    if isinstance(x, StructuredArray):
        cols = x.leaf_columns()
        labels = [c[0] for c in cols]
        tensors = [c[1] for c in cols if isinstance(c[1], torch.Tensor)]
        if tensors:
            dev = tensors[0].device
            for t in tensors:
                _check_tensor_dtype(t)
            data = torch.stack([c[1].to(dev, torch.float64) if isinstance(c[1], torch.Tensor) else
                                torch.as_tensor(numpy.asarray(c[1], dtype=numpy.float64), device=dev) for c in cols])
            return labels, data, x.shape
        data = numpy.stack([numpy.asarray(c[1], dtype=numpy.float64) for c in cols]) if cols else numpy.empty((0, x.size))
        return labels, data, x.shape
    if isinstance(x, torch.Tensor):
        _check_tensor_dtype(x)
        return [None], x.reshape(1, -1).to(torch.float64), tuple(x.shape)
    if not (numpy.issubdtype(x.dtype, numpy.number) or x.dtype == bool):
        raise TypeError(f'points have non-numerical dtype {x.dtype!r}')
    return [None], x.reshape(1, -1).astype(numpy.float64), x.shape
