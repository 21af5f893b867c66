"""``open(name, mode, **kwargs)`` factories for the format modules.

Behaviour of the reference's ``FileOpener`` (baseband/base/base.py:1650-1902):
modes 'rb', 'wb', 'rs', 'ws' ('r'/'w' default to stream mode); ``name`` is a
path or an open binary file handle; for writing, keyword arguments that are
not reader/writer options are used to build ``header0`` through
``Header.fromvalues``.  The extra stream options of this implementation
(``device``, ``chunk_nbytes``, ``dtype``) are non-header keys, so they are never fed to
the header (SURVEY.md section 5, "Config / flag system").
"""
import io
import os

__all__ = ['make_opener', 'make_info', 'normalize_mode']

COMMON_NON_HEADER = {'squeeze', 'subset', 'fill_value', 'verify',
                     'file_size', 'device', 'chunk_nbytes', 'dtype'}


def normalize_mode(mode):
    if mode in ('r', 'w'):
        mode += 's'
    if mode not in ('rb', 'wb', 'rs', 'ws'):
        raise ValueError("invalid mode {!r}; should be one of 'rb', 'wb', "
                         "'rs' or 'ws'.".format(mode))
    return mode


def make_opener(fmt, classes, header_class=None, non_header_keys=(),
                doc=None):
    """``classes``: dict mode -> class; stream classes are called as
    ``cls(fh, **kwargs)`` (writers get ``header0=``)."""
    non_header = COMMON_NON_HEADER | set(non_header_keys) | {'header0'}

    def open(name, mode='rs', **kwargs):
        mode = normalize_mode(mode)
        if mode[0] == 'w' and mode[1] == 's' and header_class is not None \
                and kwargs.get('header0') is None:
            header_kwargs = {k: kwargs.pop(k) for k in list(kwargs)
                             if k not in non_header}
            kwargs.pop('header0', None)
            sample_rate = kwargs.get('sample_rate')
            if sample_rate is not None and fmt == 'vdif':
                header_kwargs.setdefault('sample_rate', sample_rate)
            kwargs['header0'] = header_class.fromvalues(**header_kwargs)
        file_size = kwargs.pop('file_size', None)
        from ..helpers.sequentialfile import FileNameSequencer
        if isinstance(name, (tuple, list, FileNameSequencer)) or (
                isinstance(name, str) and '{' in name and mode[0] == 'w'):
            # a sequence of files (or a name template) as one byte stream
            from ..helpers import sequentialfile
            fh = sequentialfile.open(name, mode[0] + 'b',
                                     file_size=file_size)
            opened = True
        elif isinstance(name, (str, bytes, os.PathLike)):
            # writers get 'w+b' so that payloads can be memory mapped
            # (base/base.py:1763-1766)
            fh = io.open(name, 'w+b' if mode[0] == 'w' else 'rb')
            opened = True
        else:
            fh, opened = name, False
        try:
            return classes[mode](fh, **kwargs)
        except Exception:
            if opened:
                fh.close()
            raise

    open.__name__ = 'open'
    open.__doc__ = doc or 'Open a {} file for reading or writing.'.format(fmt)
    return open


class FormatInfo:
    """Minimal stand-in for the reference's ``info`` objects
    (baseband/base/file_info.py): truthy if the file looks like ``format``;
    for readable streams also carries the basic stream properties."""

    def __init__(self, format, ok, **attrs):
        self.format = format if ok else None
        self._ok = bool(ok)
        self.__dict__.update(attrs)

    def __bool__(self):
        return self._ok

    def __repr__(self):
        keys = [k for k in self.__dict__ if not k.startswith('_')]
        return '\n'.join('{} = {}'.format(k, getattr(self, k)) for k in keys)


def make_info(fmt):
    """``info(name, **kwargs)`` for a format module: the entry-point group
    ``baseband.io`` expects ``open`` and ``info`` (io/__init__.py:139-154)."""

    def info(name, **kwargs):
        from .. import guess_format
        try:
            ok = guess_format(name) == fmt
        except (OSError, TypeError):
            ok = False
        attrs = {}
        if ok:
            import importlib
            module = importlib.import_module('baseband_b200.' + fmt)
            try:
                with module.open(name, 'rs', **kwargs) as fh:
                    attrs = dict(sample_rate=fh.sample_rate,
                                 sample_shape=tuple(fh.sample_shape),
                                 samples_per_frame=fh.samples_per_frame,
                                 bps=fh.bps, complex_data=fh.complex_data,
                                 shape=fh.shape, start_time=fh.start_time,
                                 stop_time=fh.stop_time, readable=True)
            except Exception as exc:     # needs more arguments, e.g. nchan
                attrs = dict(readable=False, errors={'open': str(exc)})
        return FormatInfo(fmt, ok, **attrs)

    info.__name__ = 'info'
    return info
