"""Specification of a derivative of the process (reference: src/lsqfitgp/_Deriv.py).

`Deriv` parses what `GP.addx(deriv=)` and `CrossKernel.linop('diff', ...)` accept.  Any order parses; the Gram kernels
compute first derivatives only (order <= 1 on each argument), so higher orders raise NotImplementedError where they are
used.
"""

import collections
import numbers

__all__ = ['Deriv']


class Deriv:
    """Specification of a derivative.

    Accepted forms:
      0, None, {}   no derivative
      n (int)       n derivatives w.r.t. the single coordinate of unstructured points ("implicit")
      'a'           first derivative w.r.t. the field 'a'
      ['a', 'b']    each occurrence of a name counts once
      {'a': n}      n derivatives w.r.t. field 'a'

    `order` is the total order, `implicit` tells the integer form, iteration yields (field, order) pairs (field None
    for the implicit form). """

    def __new__(cls, *args):
        if len(args) == 1 and isinstance(args[0], Deriv):
            return args[0]
        if len(args) > 1:
            raise ValueError(f'Deriv takes one argument, got {len(args)}')
        arg = args[0] if args else None
        self = object.__new__(cls)
        self._implicit = False
        self._counter = collections.Counter()
        if arg is None:
            pass
        elif isinstance(arg, numbers.Integral) and not isinstance(arg, bool):
            if arg < 0:
                raise ValueError(f'degree {arg} < 0')
            if arg:
                self._implicit = True
                self._counter[None] = int(arg)
        elif isinstance(arg, str):
            self._counter[arg] = 1
        elif isinstance(arg, dict):
            for k, v in arg.items():
                if not isinstance(k, str):
                    raise TypeError(f'derivative field must be a string, got {k!r}')
                if not isinstance(v, numbers.Integral) or isinstance(v, bool):
                    raise TypeError(f'derivative order must be an integer, got {v!r}')
                if v < 0:
                    raise ValueError(f'degree {v} < 0')
                if v:
                    self._counter[k] = int(v)
        elif isinstance(arg, (list, tuple)):
            for k in arg:
                if not isinstance(k, str):
                    raise TypeError(f'derivative field must be a string, got {k!r}')
                self._counter[k] += 1
        else:
            raise TypeError(f'cannot interpret {arg!r} as a derivative specification')
        return self

    def __iter__(self):
        return iter(self._counter.items())

    def __bool__(self):
        return bool(self._counter)

    def __getitem__(self, field):
        return self._counter.get(field, 0)

    def __eq__(self, other):
        if not isinstance(other, Deriv):
            other = Deriv(other)
        return self._implicit == other._implicit and self._counter == other._counter

    def __hash__(self):
        return hash((self._implicit, frozenset(self._counter.items())))

    def __repr__(self):
        if self._implicit:
            return f'Deriv({self.order})'
        return f'Deriv({dict(self._counter)!r})'

    @property
    def implicit(self):
        """ True for the integer form (derivative w.r.t. the coordinate of unstructured points) """
        return self._implicit

    @property
    def order(self):
        """ total order of the derivative """
        return sum(self._counter.values())
