"""EnsembleState -- the ensemble-state object of efa_xray (efa_xray/state/ensemble.py:15-273).

The reference subclasses xarray.Dataset.  xarray cannot be installed in this image, so the class is
built on a small labelled container that exposes exactly the surface the reference and its users touch
(SURVEY.md section 8b): from_vardict(vardict, coorddict), .coords[k], .variables[k] / .keys(),
state[k].values / .shape / [y, x].values, to_array(), transpose(...), update(ds), mean(dim='mem'),
state - state.  When xarray IS importable, from_xarray()/to_xarray() convert losslessly.

Variables have dims (validtime, y, x, mem) with mem last; lat/lon are 2-D (y, x) coordinates; the state
vector layout is var -> time -> y -> x with members contiguous (ensemble.py:110-114).

Methods that do arithmetic over the grid (nearest_points, interpolate, distance_to_point) run on the GPU
through libefa_xray_b200; the scalar haversine is plain Python.
"""
from __future__ import print_function

import json
import weakref
from collections import OrderedDict
from copy import deepcopy

import numpy as np

import efa_xray_b200 as _pkg
from .. import _lib

_COORD_NAMES = ['validtime', 'lat', 'lon', 'mem', 'x', 'y']
_STATE_DIMS = ('validtime', 'y', 'x', 'mem')


class _BlockPool(object):
    """Page-locked host blocks for ensemble data.  The analysis reads the prior straight out of the state's block and
    writes the posterior straight into a new one (no staging copies), which needs page-locked memory to be
    asynchronous; cudaHostAlloc costs ~0.2 s per GB, so blocks of states that were garbage-collected are kept for
    the next analysis of the same size (cycling).  Without a CUDA device the blocks are plain numpy arrays."""

    def __init__(self, max_cached_bytes=16 << 30):
        self.free = {}            # (nbytes) -> [torch uint8 tensors]
        self.cached = 0
        self.max_cached = max_cached_bytes

    def alloc(self, shape, dtype):
        """-> (ndarray of that shape, owner): `owner` is the torch tensor to hand back to release() (or None)."""
        dtype = np.dtype(dtype)
        nbytes = int(np.prod(shape)) * dtype.itemsize
        try:
            import torch
            cuda = torch.cuda.is_available()
        except ImportError:
            cuda = False
        if not cuda or nbytes == 0:
            return np.empty(shape, dtype=dtype), None
        lst = self.free.get(nbytes)
        if lst:
            owner = lst.pop()
            self.cached -= nbytes
        else:
            owner = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
        return owner.numpy().view(dtype).reshape(shape), owner

    def release(self, owner):
        if owner is None:
            return
        nbytes = owner.numel()
        if self.cached + nbytes <= self.max_cached:
            self.free.setdefault(nbytes, []).append(owner)
            self.cached += nbytes


BLOCK_POOL = _BlockPool()


class Variable(object):
    """dims + ndarray with the .values/.shape/indexing surface of an xarray DataArray."""

    def __init__(self, dims, values):
        if isinstance(dims, str):
            dims = (dims,)
        self.dims = tuple(dims)
        self._values = np.asarray(values)
        if self._values.ndim != len(self.dims):
            raise ValueError('dims %r do not match array of shape %r' % (self.dims, self._values.shape))

    @property
    def values(self):
        return self._values

    @values.setter
    def values(self, new):
        new = np.asarray(new)
        if new.shape != self._values.shape:
            raise ValueError('replacement data must match the Variable\'s shape')
        self._values = new

    @property
    def shape(self):
        return self._values.shape

    def __len__(self):
        return self._values.shape[0]

    def __array__(self, dtype=None, copy=None):
        return np.asarray(self._values, dtype=dtype)

    def __getitem__(self, key):
        out = self._values[key]
        keys = key if isinstance(key, tuple) else (key,)
        dims, k = [], 0
        for d in self.dims:
            if k < len(keys):
                if isinstance(keys[k], slice):
                    dims.append(d)
                k += 1
            else:
                dims.append(d)
        return Variable(tuple(dims), out) if np.ndim(out) == len(dims) else out

    def __setitem__(self, key, val):
        self._values[key] = val.values if isinstance(val, Variable) else val

    def transpose(self, *dims):
        order = [self.dims.index(d) for d in dims if d in self.dims]
        return Variable(tuple(self.dims[i] for i in order), self._values.transpose(order))

    def mean(self, dim=None):
        ax = self.dims.index(dim)
        return Variable(tuple(d for d in self.dims if d != dim), self._values.mean(axis=ax))

    def _binary(self, other, op):
        if isinstance(other, Variable):
            idx = tuple(slice(None) if d in other.dims else None for d in self.dims)
            return Variable(self.dims, op(self._values, other.values[idx]))
        return Variable(self.dims, op(self._values, other))

    def __sub__(self, o):
        return self._binary(o, np.subtract)

    def __add__(self, o):
        return self._binary(o, np.add)

    def __mul__(self, o):
        return self._binary(o, np.multiply)


class _StackedArray(Variable):
    """Result of to_array(): dims ('variable', validtime, y, x, mem) plus the variable names."""

    def __init__(self, dims, values, names, coords):
        Variable.__init__(self, dims, values)
        self.names = list(names)
        self._coords = coords

    def to_dataset(self, dim='variable'):
        ds = _LabelledDataset()
        ds._coords = self._coords
        for i, n in enumerate(self.names):
            ds._data_vars[n] = Variable(self.dims[1:], self._values[i])
        return ds


class _View(object):
    def __init__(self, *dicts):
        self._dicts = dicts

    def __getitem__(self, k):
        for d in self._dicts:
            if k in d:
                return d[k]
        raise KeyError(k)

    def __contains__(self, k):
        return any(k in d for d in self._dicts)

    def __iter__(self):
        return iter(self.keys())

    def __len__(self):
        return len(self.keys())

    def keys(self):
        out = []
        for d in self._dicts:
            out.extend(d.keys())
        return out

    def items(self):
        return [(k, self[k]) for k in self.keys()]


class _LabelledDataset(object):
    """The slice of xarray.Dataset behaviour that efa_xray relies on."""

    def __init__(self, data_vars=None, coords=None):
        self._data_vars = OrderedDict()
        self._coords = OrderedDict()
        for k, v in (coords or {}).items():
            self._coords[k] = Variable(v[0], v[1]) if isinstance(v, tuple) else Variable((k,), v)
        for k, v in (data_vars or {}).items():
            self._data_vars[k] = v if isinstance(v, Variable) else Variable(v[0], v[1])

    @property
    def coords(self):
        return _View(self._coords)

    @property
    def variables(self):
        return _View(self._data_vars, self._coords)

    @property
    def data_vars(self):
        return _View(self._data_vars)

    def keys(self):
        return self.variables.keys()

    def __getitem__(self, k):
        return self.variables[k]

    def __contains__(self, k):
        return k in self.variables

    def _like(self):
        new = self.__class__.__new__(self.__class__)
        _LabelledDataset.__init__(new)
        return new

    def __deepcopy__(self, memo):
        new = self._like()
        new._data_vars = OrderedDict((k, Variable(v.dims, v.values.copy())) for k, v in self._data_vars.items())
        new._coords = OrderedDict((k, Variable(v.dims, v.values.copy())) for k, v in self._coords.items())
        if hasattr(new, '_consolidate'):
            new._consolidate()
        return new

    def copy(self, deep=True):
        return deepcopy(self) if deep else self

    def to_array(self):
        names = list(self._data_vars.keys())
        first = self._data_vars[names[0]]
        for n in names:
            if self._data_vars[n].dims != first.dims:
                raise ValueError('to_array needs all variables on the same dims')
        return _StackedArray(('variable',) + first.dims,
                             np.stack([self._data_vars[n].values for n in names], axis=0), names, self._coords)

    def transpose(self, *dims):
        new = self._like()
        new._coords = OrderedDict((k, v.transpose(*dims)) for k, v in self._coords.items())
        new._data_vars = OrderedDict((k, v.transpose(*dims)) for k, v in self._data_vars.items())
        return new

    def update(self, other):
        for k, v in other._data_vars.items():
            self._data_vars[k] = v

    def mean(self, dim=None):
        new = self._like()
        new._coords = OrderedDict((k, v) for k, v in self._coords.items() if dim not in v.dims)
        new._data_vars = OrderedDict((k, v.mean(dim=dim)) for k, v in self._data_vars.items())
        return new

    def _binary(self, other, op):
        new = self._like()
        new._coords = self._coords
        for k, v in self._data_vars.items():
            o = other._data_vars[k] if isinstance(other, _LabelledDataset) else other
            new._data_vars[k] = v._binary(o, op)
        return new

    def __sub__(self, o):
        return self._binary(o, np.subtract)

    def __add__(self, o):
        return self._binary(o, np.add)

    def __mul__(self, o):
        return self._binary(o, np.multiply)


class EnsembleState(_LabelledDataset):
    """Define an ensemble state vector (efa_xray/state/ensemble.py:15).

    Storage: when every variable has dims (validtime, y, x, mem) and the same dtype, the data of all variables lives
    in ONE contiguous block [nvar, ntimes, ny, nx, nmem] (page-locked when a CUDA device is present) and the
    variables are views into it.  That block IS the reference's state-vector layout (ensemble.py:110-114), so
    to_vect() is a reshape, the analysis uploads straight from it, and the posterior state adopts the buffer the
    analysis was downloaded into."""

    @classmethod
    def from_vardict(cls, vardict, coorddict):
        """ensemble.py:25-36.  vardict: {name: (dims, array)}; coorddict: {name: array | (dims, array)}."""
        new = cls.__new__(cls)
        _LabelledDataset.__init__(new, vardict, coorddict)
        new._consolidate()
        return new

    # ---- contiguous block -------------------------------------------------------------------------------
    def _block_view(self):
        """The [nvar, nt, ny, nx, nmem] block if every variable is still a view into it (in order), else None."""
        blk = self.__dict__.get('_block')
        if blk is None or len(self._data_vars) != blk.shape[0]:
            return None
        base = blk.__array_interface__['data'][0]
        step = blk[0].nbytes
        for i, v in enumerate(self._data_vars.values()):
            a = v._values
            if (v.dims != _STATE_DIMS or a.shape != blk.shape[1:] or a.dtype != blk.dtype or not a.flags.c_contiguous
                    or a.__array_interface__['data'][0] != base + i * step):
                return None
        return blk

    def _adopt_block(self, blk, owner=None):
        """Make the variables views of blk [nvar, nt, ny, nx, nmem] (no copy); owner = pool token of the block."""
        names = list(self._data_vars.keys())
        assert blk.shape[0] == len(names)
        for i, n in enumerate(names):
            self._data_vars[n] = Variable(_STATE_DIMS, blk[i])
        self.__dict__['_block'] = blk
        if owner is not None:
            # hand the page-locked block back to the pool when this state object goes away
            self.__dict__['_block_finalizer'] = weakref.finalize(self, BLOCK_POOL.release, owner)

    def _consolidate(self):
        """Gather the variables into one contiguous block (adopting the caller's memory when it already is one)."""
        if self._block_view() is not None:
            return True
        vs = list(self._data_vars.values())
        if not vs or any(v.dims != _STATE_DIMS for v in vs) or len({v._values.shape for v in vs}) != 1 \
                or len({v._values.dtype for v in vs}) != 1 or vs[0]._values.dtype not in (np.float64, np.float32):
            self.__dict__['_block'] = None
            return False
        first = vs[0]._values
        step = first.nbytes
        base = first.__array_interface__['data'][0]
        if step > 0 and all(v._values.flags.c_contiguous and v._values.__array_interface__['data'][0] == base + i * step
                            for i, v in enumerate(vs)):
            # the caller's arrays are consecutive slices of one buffer (e.g. block[v] views): adopt it as it is
            blk = np.lib.stride_tricks.as_strided(first, shape=(len(vs),) + first.shape, strides=(step,) + first.strides)
            self.__dict__['_block_keepalive'] = [v._values for v in vs]
            self._adopt_block(blk)
            return True
        blk, owner = BLOCK_POOL.alloc((len(vs),) + first.shape, first.dtype)
        for i, v in enumerate(vs):
            blk[i] = v._values
        self._adopt_block(blk, owner)
        return True

    def _new_with_block(self, blk, owner=None):
        """A new state with this state's coordinates (copied) and variable names whose data is blk (adopted)."""
        new = self._like()
        new._coords = OrderedDict((k, Variable(v.dims, v.values.copy())) for k, v in self._coords.items())
        new._data_vars = OrderedDict((k, None) for k in self._data_vars.keys())
        new._adopt_block(blk, owner)
        return new

    @classmethod
    def from_xarray(cls, ds):
        """Build from an xarray.Dataset (when xarray is installed)."""
        vardict = {k: (tuple(ds[k].dims), np.asarray(ds[k].values)) for k in ds.data_vars}
        coorddict = {k: (tuple(ds.coords[k].dims), np.asarray(ds.coords[k].values)) for k in ds.coords}
        return cls.from_vardict(vardict, coorddict)

    def to_xarray(self):
        import xarray
        return xarray.Dataset({k: (v.dims, v.values) for k, v in self._data_vars.items()},
                              coords={k: (v.dims, v.values) for k, v in self._coords.items()})

    # ---- sizes, ensemble.py:40-56
    def nmems(self):
        return len(self.coords['mem'])

    def ny(self):
        return len(self.coords['y'])

    def nx(self):
        return len(self.coords['x'])

    def ntimes(self):
        return len(self.coords['validtime'])

    def vars(self):
        return [x for x in self.variables.keys() if x not in _COORD_NAMES]

    def nvars(self):
        return len(self.vars())

    def nstate(self):
        return self.ntimes() * self.ny() * self.nx() * self.nvars()

    def shape(self):
        """Full shape (nvars, ntimes, ny, nx, nmems) of the stacked array."""
        blk = self._block_view()
        if blk is not None:
            return blk.shape
        return self.to_array().shape

    # ---- vector form, ensemble.py:110-121
    def to_vect(self):
        """Nstate x Nmems array, row order var -> validtime -> y -> x.  When the state's data is one contiguous
        block this is a READ-ONLY VIEW of it (no copy; take .copy() to get a private array, as the reference's
        to_vect returns); otherwise the variables are stacked as in the reference."""
        blk = self._block_view()
        if blk is not None:
            v = blk.reshape(self.nstate(), self.nmems())
            v = v.view()
            v.flags.writeable = False
            return v
        return np.reshape(self.transpose('validtime', 'y', 'x', 'mem').to_array().values,
                          (self.nstate(), self.nmems()))

    def from_vect(self, instate):
        """Takes an Nstate x Nmems ndarray and updates the state accordingly."""
        blk = self._block_view()
        if blk is not None:
            np.copyto(blk, np.reshape(instate, blk.shape))
            return
        instate = np.reshape(instate, self.shape())
        statearr = self.to_array()
        statearr.values = instate
        self.update(statearr.to_dataset(dim='variable'))
        self._consolidate()

    def ensemble_mean(self):
        return self.mean(dim='mem')

    def ensemble_perts(self):
        return self - self.ensemble_mean()

    def ensemble_times(self):
        return self['validtime'].values

    # ---- geometry on the GPU
    def _grid_tables(self):
        import torch
        from ..engine import GridTables
        lat, lon = self['lat'].values, self['lon'].values
        key = (id(lat), id(lon))
        cached = getattr(self, '_grid_cache', None)
        if cached is None or cached[0] != key:
            _lib.require_device()
            cached = (key, GridTables(lat, lon, torch.device('cuda', torch.cuda.current_device()), ny=self.ny()))
            object.__setattr__(self, '_grid_cache', cached)
        return cached[1]

    def nearest_points(self, lat, lon, npt=1):
        """Indices (y, x) of the npt grid points nearest to (lat, lon) under the reference's
        pseudo-metric hypot(dsin(lat), dcos(lon)) (ensemble.py:152-168); ties go to the lowest flat index."""
        from ..engine import stencil_search, pseudo_distance_order
        if npt > 4:
            # any npt (ensemble.py:165 takes the first npt of a full argsort): pseudo-distances of all points on
            # the device, stable sort there (ties -> lowest flat index)
            flat = pseudo_distance_order(self._grid_tables(), float(lat), float(lon), int(npt))
        else:
            idx4, _, _ = stencil_search(self._grid_tables(), np.array([lat], dtype=np.float64),
                                        np.array([lon], dtype=np.float64))
            flat = idx4.cpu().numpy()[0, :npt]
        return np.unravel_index(flat, self['lat'].shape)

    def interpolate(self, var, time, lat, lon, forward_operator='reference'):
        """Ensemble estimate [nmems] of `var` at (time, lat, lon): 4-point inverse-distance weights in
        space x linear weights in time (ensemble.py:170-239, weights as the reference computes them).
        forward_operator='bilinear' (2-D lat/lon only) interpolates bilinearly on the grid cell that contains the
        point and linearly in time with correctly oriented weights (DESIGN.md section 4.8); a point outside the grid
        raises ValueError."""
        from ..engine import ObsArrays, ob_priors, time_weights, check_forward_operator
        import torch
        check_forward_operator(forward_operator, np.ndim(self['lat'].values))
        tlo, thi, wlo, whi, outside = time_weights(self['validtime'].values, np.array([np.datetime64(time)]),
                                                   swapped=forward_operator == 'reference')
        if outside[0]:
            print("Interpolation is outside of time range in state!")
            return None
        grid = self._grid_tables()
        vals = np.ascontiguousarray(self.variables[var].values)
        nt, ny, nx, nmem = vals.shape
        X = torch.from_numpy(vals.reshape(nt * ny * nx, nmem)).to(grid.device)
        obs = ObsArrays(value=np.zeros(1), error=np.ones(1), lat=np.array([lat], dtype=np.float64),
                        lon=np.array([lon], dtype=np.float64), halfwidth=np.ones(1),
                        assimilate=np.zeros(1, dtype=np.uint8), row0=tlo * ny * nx, row1=thi * ny * nx,
                        tw0=wlo, tw1=whi)
        Y, nex = ob_priors(X, grid, obs, 'f64' if X.dtype == torch.float64 else 'f32', forward_operator=forward_operator)
        if forward_operator == 'bilinear':
            if int(nex.item()) > 0:
                raise ValueError('(%r, %r) lies outside the grid: the bilinear forward operator has no cell to '
                                 'interpolate from' % (lat, lon))
        elif int(nex.item()) > 0 and _pkg.EXACT_MATCH_POLICY == 'raise':
            raise IndexError('observation within 1 km of a grid point: the reference raises here '
                             '(state/ensemble.py:195-196); set efa_xray_b200.EXACT_MATCH_POLICY = "nearest" '
                             'to use the nearest point instead')
        out = Y[0].cpu().numpy().astype(np.float64)
        # the reference's 1-D lat/lon branch returns the estimate with a leading axis of length 1 (ensemble.py:233-234)
        return out[None, :] if grid.diag else out

    def haversine(self, loc1, loc2):
        """Great-circle distance in km between two (lat, lon) pairs (ensemble.py:241-252)."""
        from ..observation.observation import haversine
        return haversine(loc1, loc2)

    def distance_to_point(self, lat, lon):
        """Haversine distance in km from every grid point to (lat, lon) (ensemble.py:254-267)."""
        import torch
        grid = self._grid_tables()
        u, n = (grid.u1, grid.nx) if grid.diag else (grid.u, grid.npts)
        out = torch.empty(n, dtype=torch.float64, device=grid.device)
        _lib.call('exb_localization_weights', _lib.ptr(u), n, float(lat), float(lon), 1.0, 0,
                  _lib.ptr(out), None, _lib.stream_ptr())
        return out.cpu().numpy().reshape(self['lat'].shape)

    def save_to_disk(self, filename='ens_state.nc'):
        """ensemble.py:269-273.  netCDF through xarray when it is installed, otherwise a .npz archive with
        the same variables and coordinates."""
        try:
            self.to_xarray().to_netcdf(filename)
        except ImportError:
            arrays = {'var__' + k: v.values for k, v in self._data_vars.items()}
            arrays.update({'coord__' + k: v.values for k, v in self._coords.items()})
            arrays['__dims__'] = np.array(json.dumps({k: list(v.dims) for k, v in self.variables.items()}))
            with open(filename, 'wb') as f:          # exactly this file name (np.savez(name) would append .npz)
                np.savez(f, **arrays)

    @classmethod
    def load_from_disk(cls, filename):
        """Inverse of the .npz branch of save_to_disk."""
        with np.load(filename, allow_pickle=False) as z:
            dims = json.loads(str(z['__dims__']))
            if not (isinstance(dims, dict) and all(isinstance(k, str) and isinstance(v, list) and
                                                   all(isinstance(d, str) for d in v) for k, v in dims.items())):
                raise ValueError('%s: malformed __dims__ record' % (filename,))
            dims = {k: tuple(v) for k, v in dims.items()}
            vardict = {k[5:]: (dims[k[5:]], z[k]) for k in z.files if k.startswith('var__')}
            coorddict = {k[7:]: (dims[k[7:]], z[k]) for k in z.files if k.startswith('coord__')}
        return cls.from_vardict(vardict, coorddict)
