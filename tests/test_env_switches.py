"""The environment variables the library reads are exactly the supported switches listed in README.md.  Each one is read once
per process and silently changes which kernel or schedule runs, so a new one has to be a deliberate, documented choice.
Source scan only: needs neither the library nor a GPU."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PACKAGE = os.path.join(ROOT, 'nnr_b200')

SUPPORTED = {'NNR_GEMM_ALGO', 'NNR_LSTM_ALGO', 'NNR_LANES', 'NNR_LSTM_DEBUG', 'NNR_B200_LIB'}

# getenv("X") in C / CUDA, os.environ.get('X'), os.environ['X'] and os.getenv('X') in Python
_READ = re.compile(r'''(?:getenv\s*\(|environ\s*\.\s*get\s*\(|environ\s*\[)\s*["']([A-Za-z0-9_]+)["']''')


def _sources():
    for d, dirs, files in os.walk(PACKAGE):
        dirs[:] = [x for x in dirs if not x.startswith('.') and x not in ('_lib', '__pycache__')]
        for f in sorted(files):
            if f.endswith(('.py', '.cu', '.cuh', '.h', '.sh')):
                path = os.path.join(d, f)
                with open(path, encoding='utf-8') as fh:
                    yield os.path.relpath(path, ROOT), fh.read()


def test_library_reads_exactly_the_supported_switches():
    read = {}
    for rel, text in _sources():
        for name in _READ.findall(text):
            read.setdefault(name, []).append(rel)
    assert set(read) == SUPPORTED, {'unexpected': {n: read[n] for n in set(read) - SUPPORTED},
                                    'missing': sorted(SUPPORTED - set(read))}


def test_no_compile_time_prefetch_switch():
    for rel, text in _sources():
        assert 'NNR_LSTM_PFD' not in text, rel


def test_readme_names_exactly_the_supported_switches():
    with open(os.path.join(ROOT, 'README.md'), encoding='utf-8') as fh:
        readme = fh.read()
    m = re.search(r'^Environment switches:.*?(?=\n\s*\n)', readme, re.S | re.M)
    assert m, 'README.md has no "Environment switches:" paragraph'
    assert set(re.findall(r'`(NNR_[A-Z0-9_]+)', m.group(0))) == SUPPORTED
