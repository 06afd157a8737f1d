"""Kernel selection of mlb_forward without a GPU.  monoloco_b200/csrc/fwd_plan.h is plain C++17, so a small program (g++)
runs plan_forward() over a table of requests on handles with the calibrate() default wave times of a 148-SM B200
(cluster wave 0.185 ms, row-tile wave 0.42 + 0.067 TM ms, tensor-core wave 0.33 ms, 11 resident 8-CTA clusters,
33 resident tensor-core clusters)."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from monoloco_b200._lib import FWD_FORCE_CLUSTER, FWD_FORCE_TC, FWD_FORCE_TILE, FWD_FORCE_WIDE, FWD_FORCE_WIDE2  # noqa: E402

TILE, CLUSTER, WIDE, TC, WIDE2 = 0, 1, 2, 3, 4  # MLB_KERNEL_*
# the families mlb_create sets up for each hidden width
HANDLES = {1024: (TILE, CLUSTER, WIDE, TC, WIDE2), 512: (TILE, WIDE, TC, WIDE2), 384: (TILE, WIDE, WIDE2),
           256: (TILE, WIDE, TC, WIDE2), 2048: (TC,)}

DRIVER = r'''
#include <cstdio>
#include "fwd_plan.h"
int main() {
    unsigned have, disabled;
    double t_tc;
    int n_rows, flags, rpg;
    while (scanf("%u %u %lf %d %d %d", &have, &disabled, &t_tc, &n_rows, &flags, &rpg) == 6) {
        mlb::FwdPlanInputs in = {};
        in.have = have, in.disabled = disabled;
        in.t_cluster_wave = 0.185, in.t_tile_a = 0.42, in.t_tile_b = 0.067, in.t_tc_wave = t_tc;
        in.n_sms = 148, in.small_conc = 11, in.tc_clusters = 33, in.tile_ctas[0] = 148, in.tile_ctas[1] = 148;
        const mlb::FwdPlan p = mlb::plan_forward(in, n_rows, flags, rpg);
        if (p.kernel < 0) printf("error %s\n", p.error);
        else printf("%d %d %d %d %d %d\n", p.kernel, p.tm, p.grid, p.clusters, p.launches, p.arrivals);
    }
    return 0;
}
'''

# (width, rows, flags, rows_per_group, disabled kernels, tensor-core wave ms) -> kernel and the geometry it must have,
# or None for an error
CASES = [
    ((1024, 1, 0, 0, (), 0.33), (WIDE2, dict(arrivals=1))),
    ((1024, 16, 0, 0, (), 0.33), (WIDE2, dict(arrivals=1))),
    ((1024, 17, 0, 0, (), 0.33), (WIDE, dict(launches=1, arrivals=1))),
    ((1024, 33, 0, 0, (), 0.33), (WIDE, dict(launches=2, arrivals=1))),
    ((1024, 64, 0, 0, (), 0.33), (WIDE, dict(launches=2, arrivals=1))),
    ((1024, 65, 0, 0, (), 0.33), (CLUSTER, dict(clusters=5, arrivals=5))),
    ((1024, 176, 0, 0, (), 0.33), (CLUSTER, dict(clusters=11, arrivals=11))),
    ((1024, 177, 0, 0, (), 0.33), (TC, dict(clusters=2, arrivals=2))),
    ((1024, 4096, 0, 0, (), 0.33), (TC, dict(clusters=32, arrivals=32))),
    ((1024, 65536, 0, 0, (), 0.33), (TC, dict(clusters=33, arrivals=33))),
    ((1024, 16, 0, 0, (WIDE2, WIDE), 0.33), (CLUSTER, dict(clusters=1, arrivals=1))),
    ((1024, 16, FWD_FORCE_WIDE2, 0, (WIDE2,), 0.33), (WIDE2, dict(arrivals=1))),  # a forced kernel ignores the disabled bit
    ((1024, 4096, 0, 0, (), 10.0), (TILE, dict(tm=14, grid=147, arrivals=147))),
    ((256, 65, 0, 0, (), 0.33), (TC, dict(clusters=1, arrivals=1))),
    ((256, 50, 0, 0, (WIDE,), 0.33), (TILE, dict(tm=8, grid=4, arrivals=4))),
    ((384, 1000, 0, 0, (), 0.33), (TILE, dict(tm=8, grid=63, arrivals=63))),
    ((2048, 1, 0, 0, (), 0.33), (TC, dict(clusters=1, arrivals=1))),
    ((2048, 1, FWD_FORCE_TILE, 0, (), 0.33), None),
    ((2048, 1, FWD_FORCE_WIDE, 0, (), 0.33), None),
    ((2048, 1, FWD_FORCE_WIDE2, 0, (), 0.33), None),
    ((2048, 1, 0, 8, (), 0.33), None),
    ((1024, 75, FWD_FORCE_WIDE, 0, (), 0.33), (WIDE, dict(launches=3, arrivals=1))),
    ((1024, 1000, 0, 8, (), 0.33), (TILE, dict(tm=8, grid=63, arrivals=63))),
    ((1024, 10, FWD_FORCE_CLUSTER, 8, (), 0.33), (CLUSTER, dict(clusters=1, arrivals=1))),  # forced: rows_per_group ignored
    ((384, 300, FWD_FORCE_TC, 0, (), 0.33), None),
    ((512, 300, FWD_FORCE_CLUSTER, 0, (), 0.33), None),
    ((1024, 300, FWD_FORCE_TILE | FWD_FORCE_TC, 0, (), 0.33), None),
    ((1024, 8, FWD_FORCE_WIDE | FWD_FORCE_WIDE2, 0, (), 0.33), None),
    ((1024, 17, FWD_FORCE_WIDE2, 0, (), 0.33), None),
    ((384, 8, FWD_FORCE_WIDE2, 0, (WIDE2,), 0.33), (WIDE2, dict(arrivals=1))),
    ((1024, 1000, 0, 7, (), 0.33), None),
]


@pytest.fixture(scope='module')
def plans(tmp_path_factory):
    tmp = tmp_path_factory.mktemp('plan')
    src = tmp / 'plan.cpp'
    src.write_text(DRIVER)
    exe = tmp / 'plan'
    subprocess.run(['g++', '-std=c++17', '-Wall', '-Wextra', '-Werror', '-I', os.path.join(ROOT, 'monoloco_b200', 'csrc'),
                    str(src), '-o', str(exe)], check=True)
    lines = []
    for (L, rows, flags, rpg, disabled, t_tc), _ in CASES:
        have = sum(1 << k for k in HANDLES[L])
        lines.append('%d %d %r %d %d %d' % (have, sum(1 << k for k in disabled), t_tc, rows, flags, rpg))
    out = subprocess.run([str(exe)], input='\n'.join(lines) + '\n', check=True, stdout=subprocess.PIPE, text=True).stdout
    return out.splitlines()


@pytest.mark.parametrize('i', range(len(CASES)), ids=['L%d-n%d-f%d-g%d-d%s-tc%g' % (c[0][:4] + (''.join(map(str, c[0][4])) or '0', c[0][5]))
                                                       for c in CASES])
def test_plan(plans, i):
    _, want = CASES[i]
    got = plans[i]
    if want is None:
        assert got.startswith('error mlb_forward:'), got
        return
    kernel, tm, grid, clusters, launches, arrivals = map(int, got.split())
    geometry = dict(tm=tm, grid=grid, clusters=clusters, launches=launches, arrivals=arrivals)
    assert kernel == want[0], got
    for k, v in want[1].items():
        assert geometry[k] == v, (k, got)
