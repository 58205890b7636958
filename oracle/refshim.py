"""Import the REAL reference modules from /root/reference (build container only).

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  /root/reference does not exist on the
GPU box: nothing in the ``-m gpu`` tests, ``smoke()`` or ``bench.py`` calls this module.  It is
used by ``tests/golden/make_golden.py`` only (fixture generation).

How: ``bonito/__init__.py`` imports every CLI (mappy, pysam, remora, ...), so ``bonito`` is
installed as a bare namespace package whose ``__path__`` points at the reference tree; the
absent third-party modules the hot path touches at import time are stubbed:

  seqdist.{core,sparse,ctc_simple}  -> oracle.seqdist_restated   (crf/model.py:9-11)
  koi.lstm, koi.decode, parasail    -> empty stubs / restated to_str  (util.py:18-19, crf/basecall.py:9)
  numpy.int                          -> int   (crf/basecall.py:63 uses the alias removed in NumPy 1.24)
"""
import importlib
import os
import sys
import types

REFERENCE_ROOT = os.environ.get('XB_REFERENCE_ROOT', '/root/reference')
_BONITO_DIR = os.path.join(REFERENCE_ROOT, 'ub-bonito', 'bonito')


def available():
    return os.path.isfile(os.path.join(_BONITO_DIR, 'nn.py'))


def _to_str(x, encoding='ascii'):
    """koi.decode.to_str semantics as used at crf/basecall.py:90-91: drop zeros, bytes -> str."""
    import numpy as np
    x = np.asarray(x)
    return x[x.nonzero()[0]].astype('u1').tobytes().decode(encoding)


def install():
    """Install the namespace package + stubs (idempotent).  Returns the dict of loaded modules."""
    if not available():
        raise RuntimeError('reference tree not present at %s' % REFERENCE_ROOT)
    import numpy as np
    from oracle import seqdist_restated as sr

    if not hasattr(np, 'int'):
        np.int = int

    def module(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    if 'seqdist' not in sys.modules:
        pkg = module('seqdist')
        pkg.__path__ = []
        pkg.core = module('seqdist.core', SequenceDist=sr.SequenceDist, Max=sr.Max, Log=sr.Log,
                          semiring=sr.semiring)
        pkg.sparse = module('seqdist.sparse', logZ=sr.sparse.logZ,
                            fwd_scores_cupy=sr.sparse.fwd_scores_cupy,
                            bwd_scores_cupy=sr.sparse.bwd_scores_cupy)
        pkg.ctc_simple = module('seqdist.ctc_simple', logZ_cupy=sr.ctc_simple.logZ_cupy,
                                viterbi_alignments=sr.ctc_simple.viterbi_alignments)
    if 'koi' not in sys.modules:
        koi = module('koi')
        koi.__path__ = []
        koi.lstm = module('koi.lstm')
        koi.decode = module('koi.decode', beam_search=None, to_str=_to_str)
    if 'parasail' not in sys.modules:
        module('parasail')
    if 'bonito' not in sys.modules or getattr(sys.modules['bonito'], '__xb_shim__', False) is False:
        b = types.ModuleType('bonito')
        b.__path__ = [_BONITO_DIR]
        b.__xb_shim__ = True
        sys.modules['bonito'] = b
    mods = {}
    for name in ('bonito.nn', 'bonito.multiprocessing', 'bonito.util', 'bonito.crf.model',
                 'bonito.crf.basecall'):
        mods[name] = importlib.import_module(name)
    return mods


def reference_config(labels=('N', 'A', 'C', 'G', 'T', 'X'), state_len=3):
    """The sup@v3.3 config (bonito/models/xna_r9.4.1_e8_sup@v3.3/config.toml) with a chosen alphabet."""
    return {
        'global_norm': {'state_len': state_len},
        'input': {'features': 1},
        'model': {'package': 'bonito.crf'},
        'labels': {'labels': list(labels)},
        'encoder': {'stride': 5, 'activation': 'swish', 'features': 768, 'winlen': 19,
                    'scale': 5.0, 'rnn_type': 'lstm', 'blank_score': 2.0},
        'basecaller': {'batchsize': 384, 'chunksize': 3600, 'overlap': 500},
    }


def install_io():
    """Also load bonito.io and bonito.fast5 (golden fixtures for the output formats and the signal pre-processing):
    mappy / pysam / ont_fast5_api are stubbed -- only the pure-Python / numpy functions of those modules are used
    (write_fastq, summary_row, CSVLogger, Writer in 'wfq' mode; trim, med_mad, norm_by_noisiest_section)."""
    mods = install()

    def module(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    class _Anything:
        def __init__(self, *a, **k):
            pass

        @classmethod
        def from_references(cls, *a, **k):
            return cls()

    if 'mappy' not in sys.modules:
        module('mappy', __version__='0.0-stub')
    if 'pysam' not in sys.modules:
        module('pysam', AlignmentFile=_Anything, AlignmentHeader=_Anything, AlignedSegment=_Anything)
    if 'ont_fast5_api' not in sys.modules:
        pkg = module('ont_fast5_api')
        pkg.__path__ = []
        module('ont_fast5_api.fast5_interface', get_fast5_file=None)
    if 'bonito.cli' not in sys.modules:
        cli = module('bonito.cli')
        cli.__path__ = []
        module('bonito.cli.convert', typical_indices=None)
    sys.modules['bonito'].__version__ = '0.0-shim'
    for name in ('bonito.io', 'bonito.fast5'):
        mods[name] = importlib.import_module(name)
    return mods
