"""K5 (small-region removal + class counts, csrc/ccl.cu) against the oracle on the adversarial catalogue of
tests/ccl_patterns.py, bit for bit, on both labelling paths (``pytest -m gpu``).

Every group of entries of one shape and threshold runs as a dense batch between guard images and as a ragged canvas
with random bytes below each image, each four times on a dirty workspace (tests/ccl_pixel_worker.py).  The run kernels
(every width up to 1024) run in this process; the per-pixel kernels in a child process with NBC_CCL_RUNS=0.  Each
result must equal ``oracle.postprocess.remove_small_zones`` per image, the counts its per-class bincount, and the dead
rows of a canvas must come back unchanged."""
import os
import subprocess
import sys
from collections import Counter

import numpy as np
import pytest

import ccl_patterns as P
from ccl_pixel_worker import run_job
from oracle import postprocess as opost

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
PATHS = ('runs', 'pixels')


def _expected_dense(batch, threshold):
    memo = {}
    out = []
    for img in batch:
        key = img.tobytes()
        if key not in memo:
            memo[key] = opost.remove_small_zones_2d(img, threshold)
        out.append(memo[key])
    exp = np.stack(out)
    counts = np.stack([np.bincount(e.ravel(), minlength=3)[:3] for e in exp])
    return exp, counts


@pytest.fixture(scope='module')
def suite():
    cases = P.catalogue()
    jobs = []
    for (H, W, T), entries in P.groups(cases).items():
        batch = P.dense_batch(entries)
        exp, counts = _expected_dense(batch, T)
        place = [1 + 2 * j for j in range(len(entries))] if len(entries) > 1 else [1, 3]
        owners = [None] * len(batch)
        for j, n in enumerate(place):
            owners[n] = j if len(entries) > 1 else 0
        jobs.append(dict(kind='dense', entries=entries, canvas=batch, heights=None, T=T, exp=exp, counts=counts,
                         owners=owners))
        canvas, heights, owners = P.ragged_canvas(entries, seed=len(jobs))
        exp, counts = P.ragged_expected(canvas, heights, T)
        jobs.append(dict(kind='ragged', entries=entries, canvas=canvas, heights=heights, T=T, exp=exp, counts=counts,
                         owners=owners))
    return dict(cases=cases, jobs=jobs, got={})


def _check(job, mask, counts, problems):
    """Failure messages for one job's result."""
    msgs = ['%s %s: %s' % (job['kind'], job['entries'][0].name, p) for p in problems]
    if not np.array_equal(mask, job['exp']):
        # every entry whose own image is wrong, by name: which families a defect shows up in
        for n in sorted({int(i) for i in np.nonzero((mask != job['exp']).any(axis=(1, 2)))[0]}):
            if job['owners'][n] is not None:
                msgs.append('%s %s: wrong' % (job['kind'], job['entries'][job['owners'][n]].name))
        n, y, x = np.argwhere(mask != job['exp'])[0]
        j = job['owners'][n]
        who = 'guard image' if j is None else job['entries'][j].name
        msgs.append('%s %s (T=%d): %d bytes differ from the oracle, first in image %d at (%d, %d), got %d expected %d'
                    % (job['kind'], who, job['T'], int((mask != job['exp']).sum()), n, y, x, mask[n, y, x],
                       job['exp'][n, y, x]))
    if not np.array_equal(counts, job['counts']):
        msgs.append('%s %s: class counts %s, expected %s' % (job['kind'], job['entries'][0].name,
                                                            counts.tolist()[:4], job['counts'].tolist()[:4]))
    return msgs


def _summary(failures):
    wrong = Counter(m.split()[1].split('/')[0] for m in failures if m.endswith(': wrong'))
    return '%d failures, wrong entries by family %s:\n%s' % (len(failures), dict(wrong), '\n'.join(
        [m for m in failures if not m.endswith(': wrong')][:20]))


def test_run_path_equals_oracle(suite, cuda_device):
    if os.environ.get('NBC_CCL_RUNS', '1') not in ('', '1'):
        pytest.skip('NBC_CCL_RUNS selects the per-pixel kernels in this process')
    got, failures = [], []
    for job in suite['jobs']:
        mask, counts, problems = run_job(job['canvas'], job['heights'], job['T'], cuda_device)
        failures += _check(job, mask, counts, problems)
        got.append(mask)
    suite['got']['runs'] = got
    assert not failures, _summary(failures)


def test_pixel_path_equals_oracle(suite, cuda_device, tmp_path):
    jobs = {'count': np.array(len(suite['jobs']))}
    for k, job in enumerate(suite['jobs']):
        jobs['canvas%d' % k], jobs['threshold%d' % k] = job['canvas'], np.array(job['T'])
        if job['heights'] is not None:
            jobs['heights%d' % k] = job['heights']
    src, dst = str(tmp_path / 'jobs.npz'), str(tmp_path / 'results.npz')
    np.savez(src, **jobs)
    del jobs
    env = dict(os.environ, NBC_CCL_RUNS='0')
    r = subprocess.run([sys.executable, os.path.join(HERE, 'ccl_pixel_worker.py'), src, dst], env=env,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    res = np.load(dst)
    got, failures = [], []
    for k, job in enumerate(suite['jobs']):
        mask = res['mask%d' % k]
        failures += _check(job, mask, res['counts%d' % k], [str(p) for p in res['problems%d' % k]])
        got.append(mask)
    suite['got']['pixels'] = got
    assert not failures, _summary(failures)


def test_int64_drop_in_per_family(suite, cuda_device):
    """utils.remove_small_zones (int64, in place, returns its argument) on the first entry of every family."""
    import torch
    from neuralbarkcalculator_b200 import utils
    for family in P.FAMILIES:
        case = next(c for c in suite['cases'] if c.family == family)
        t = torch.from_numpy(case.mask.astype(np.int64)).unsqueeze(0).to(cuda_device)
        r = utils.remove_small_zones(t, case.threshold)
        assert r is t, family
        assert np.array_equal(t[0].cpu().numpy(), opost.remove_small_zones_2d(case.mask.astype(np.int64), case.threshold)), \
            case.name


def test_report_and_wrong_references(suite):
    """One line per family, then every wrong reference of ccl_patterns must disagree with the KERNEL's output on the
    entry written for it, on both paths."""
    missing = [p for p in PATHS if p not in suite['got']]
    if missing:
        pytest.fail('no kernel results for %s: run the whole module' % ', '.join(missing))
    comps = {c.name: P.components(c.mask) for c in suite['cases']}
    stats = {f: dict(cases=0, components=0, pixels=0, widths=set(), kinds=set()) for f in P.FAMILIES}
    for c in suite['cases']:
        stats[c.family]['cases'] += 1
        stats[c.family]['components'] += comps[c.name]
    for job in suite['jobs']:
        N, H, W = job['canvas'].shape
        for n, j in enumerate(job['owners']):
            if j is None:
                continue
            s = stats[job['entries'][j].family]
            s['pixels'] += (H if job['heights'] is None else int(job['heights'][n])) * W
            s['widths'].add(W)
            s['kinds'].add(job['kind'])
    print()
    for f in P.FAMILIES:
        s = stats[f]
        print('K5 %-10s cases %4d  components %8d  pixels %10d per path x 4 dirty workspaces  widths %s  %s  paths %s'
              % (f, s['cases'], s['components'], s['pixels'], sorted(s['widths']), '+'.join(sorted(s['kinds'])),
                 'default + NBC_CCL_RUNS=0'))
        assert s['kinds'] == {'dense', 'ragged'}, f
    widths = set().union(*(s['widths'] for s in stats.values()))
    assert set(P.WIDTHS + P.PIXEL_WIDTHS) <= widths

    index = {}
    for k, job in enumerate(suite['jobs']):
        for n, j in enumerate(job['owners']):
            if j is not None:
                index.setdefault((job['entries'][j].name, job['kind']), (k, n))
    cases = {c.name: c for c in suite['cases']}
    for control, (name, how) in P.CONTROLS.items():
        case = cases[name]
        k, n = index[(name, 'ragged' if how == 'ragged' else 'dense')]
        job = suite['jobs'][k]
        for path in PATHS:
            got = suite['got'][path][k]
            if how == 'image':
                assert not np.array_equal(P.wrong_output(control, case, None), got[n]), (control, path)
            elif how == 'dense':
                assert not np.array_equal(P.wrong_output(control, case, job['canvas']), got), (control, path)
            else:
                assert not np.array_equal(P.wrong_output(control, case, (job['canvas'], job['heights'])), got), \
                    (control, path)
