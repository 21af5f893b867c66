"""The drop-in boundary as the reference's plug-in loaders see it.

``baseband.io`` (baseband/io/__init__.py:35-94) resolves a format name
through an ``importlib.metadata.EntryPoint`` of group 'baseband.io' that
points to a module, loads it, and calls ``module.open(name, mode=...,
**kwargs)`` (:236-237) and ``module.info(name, **kwargs)`` (:163-164);
``baseband.tasks`` (baseband/tasks/__init__.py:25-62) does the same for
functions of group 'baseband.tasks'.  Here the entry points pyproject.toml
declares are installed as a distribution's metadata in a temporary
directory, found through ``importlib.metadata.entry_points(group=...)`` as
those loaders find them, loaded, and files are opened and read through them.
"""
import os
import tomllib
from importlib.metadata import EntryPoint, entry_points

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, sample_path

OUT = np.load(os.path.join(GOLDEN, 'sample_outputs.npz'))
FORMATS = ('vdif', 'mark5b', 'mark4', 'dada', 'guppi', 'gsb')


def _read_all_through(open_, tag=''):
    """Open and read every sample format through ``open_(name, mode,
    format, **kwargs)``; compare with the reference's outputs (golden)."""
    with open_(sample_path('sample.vdif'), 'rs', 'vdif' + tag) as fh:
        data = fh.read()
    assert np.array_equal(data, OUT['sample_vdif_data'][:, :, 0])
    with open_(sample_path('sample.m5b'), 'rs', 'mark5b' + tag, nchan=8,
               kday=56000, sample_rate=32e6) as fh:
        assert np.array_equal(fh.read(), OUT['sample_m5b_data'])
    with open_(sample_path('sample.m4'), 'rs', 'mark4' + tag, ntrack=64,
               decade=2010, sample_rate=32e6, fill_value=-7.) as fh:
        assert np.array_equal(fh.read(), OUT['sample_m4_data'])
    with open_(sample_path('sample.dada'), 'rs', 'dada' + tag,
               squeeze=False) as fh:
        assert np.array_equal(fh.read(), OUT['sample_dada_data'])
    with open_(sample_path('sample.vdif'), 'rb', 'vdif' + tag) as fb:
        assert fb.read_frame().shape == (20000, 1)


def _declared_entry_points(tmp_path, monkeypatch, group):
    """The entry points of ``group`` as an installed baseband_b200 exposes
    them: pyproject.toml's declarations written to a dist-info directory on
    sys.path, then looked up through importlib.metadata."""
    with open(os.path.join(ROOT, 'pyproject.toml'), 'rb') as fh:
        project = tomllib.load(fh)['project']
    info = tmp_path / 'baseband_b200-{}.dist-info'.format(project['version'])
    info.mkdir()
    (info / 'METADATA').write_text('Metadata-Version: 2.1\nName: {}\n'
                                   'Version: {}\n'.format(project['name'],
                                                          project['version']))
    (info / 'entry_points.txt').write_text(''.join(
        '[{}]\n'.format(name) + ''.join('{} = {}\n'.format(k, v)
                                        for k, v in eps.items())
        for name, eps in project['entry-points'].items()))
    monkeypatch.syspath_prepend(str(tmp_path))
    return {ep.name: ep for ep in entry_points(group=group)
            if ep.dist is not None and ep.dist.name == project['name']}


def test_io_entry_points_cpu(tmp_path, monkeypatch):
    import cpu_backend
    cpu_backend.install(monkeypatch)
    import baseband_b200 as bb
    eps = _declared_entry_points(tmp_path, monkeypatch, 'baseband.io')
    assert sorted(eps) == sorted(fmt + '_b200' for fmt in FORMATS)
    modules = {name: ep.load() for name, ep in eps.items()}
    for fmt in FORMATS:
        assert modules[fmt + '_b200'] is getattr(bb, fmt)
    _read_all_through(lambda name, mode, fmt, **kw:
                      modules[fmt].open(name, mode=mode, **kw), tag='_b200')
    info = modules['vdif_b200'].info(sample_path('sample.vdif'))
    assert info and info.format == 'vdif'
    assert not modules['mark5b_b200'].info(sample_path('sample.vdif'))


def test_tasks_entry_points_cpu(tmp_path, monkeypatch):
    import cpu_backend
    cpu_backend.install(monkeypatch)
    import baseband_b200 as bb
    from baseband_b200 import tasks as b200_tasks
    eps = _declared_entry_points(tmp_path, monkeypatch, 'baseband.tasks')
    assert sorted(eps) == ['integrated_power', 'moments', 'state_counts']
    tasks = {name: ep.load() for name, ep in eps.items()}
    for name, fn in tasks.items():
        assert fn is getattr(b200_tasks, name)
    with bb.vdif.open(sample_path('sample.vdif'), 'rs') as fh:
        counts = tasks['state_counts'](fh, 20000)
        data = OUT['sample_vdif_data'][:, :, 0]
        lv = b200_tasks.state_levels(fh)
        want = np.stack([np.stack([(data[b * 20000:(b + 1) * 20000] == v
                                    ).sum(0) for v in lv], -1)
                         for b in range(2)])
        assert np.array_equal(counts, want)
        fh.seek(0)
        power = tasks['integrated_power'](fh, 20000)
        ref = np.stack([(data[b * 20000:(b + 1) * 20000].astype(np.float64)
                         ** 2).mean(0) for b in range(2)])
        assert np.allclose(power, ref, rtol=1e-10, atol=0)


def test_entry_point_protocol_cpu(monkeypatch):
    import cpu_backend
    cpu_backend.install(monkeypatch)
    _entry_point_protocol()


@pytest.mark.gpu
def test_entry_point_protocol_gpu():
    _entry_point_protocol()


def _entry_point_protocol():
    """EntryPoint('<fmt>', 'baseband_b200.<fmt>', '').load() is a module with
    the ``open`` / ``info`` the loader calls; the package's own pyproject
    declares the same entry points."""
    modules = {fmt: EntryPoint(fmt, 'baseband_b200.' + fmt, '').load()
               for fmt in FORMATS}
    _read_all_through(lambda name, mode, fmt, **kw:
                      modules[fmt].open(name, mode=mode, **kw))
    info = modules['vdif'].info(sample_path('sample.vdif'))
    assert info and info.format == 'vdif'
    text = open(os.path.join(os.path.dirname(GOLDEN), '..',
                             'pyproject.toml')).read()
    assert 'baseband.io' in text
    for fmt in FORMATS:
        assert 'baseband_b200.' + fmt in text
