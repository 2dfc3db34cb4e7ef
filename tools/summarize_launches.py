"""Summarise an ncu launch list (`--metrics gpu__time_duration.sum[,dram__bytes_read.sum,dram__bytes_write.sum] --csv`):
per-kernel totals of ONE training step (the launches between the last two fused_sgd kernels) -> markdown, plus a JSON with
the DRAM traffic per bench.py kernel class (`roofline.traffic`).
usage: summarize_launches.py in.csv[.gz] out.md [title] [out.json]
A launch list named *.gz is read gzip-compressed (the test input tests/golden/r02_launches.csv.gz is the compressed
profiles/r02_launches.csv)."""
import collections
import csv
import gzip
import json
import sys


def open_text(path):
    return gzip.open(path, 'rt') if path.endswith('.gz') else open(path)


CLASSES = {   # kernel-name prefix -> class name used by bench.py (ops._T)
    'conv_wgrad': 'conv_wgrad', 'conv_halo_wgrad': 'conv_wgrad',
    'conv_igemm': 'conv_fprop+dgrad', 'conv_halo_kernel': 'conv_fprop+dgrad', 'conv_pair': 'conv_fprop+dgrad',
    'bn_apply': 'bn_apply', 'bn_bwd_dx': 'bn_bwd_dx', 'bn_bwd_reduce': 'bn_bwd_reduce', 'bn_finalize': 'bn_stats',
    'bn_stats': 'bn_stats', 'maxpool': 'pool', 'avgpool': 'pool', 'fused_sgd': 'fused_sgd',
}


def main(src, dst, title, js=None):
    with open_text(src) as f:
        lines = [l for l in f if l.startswith('"')]
    r = csv.reader(lines)
    hdr = next(r)
    ix = {h: i for i, h in enumerate(hdr)}
    launches = collections.OrderedDict()          # ID -> {name, metric: value}
    for row in r:
        if len(row) != len(hdr):
            continue
        d = launches.setdefault(row[ix['ID']], {'name': row[ix['Kernel Name']]})
        try:
            d[row[ix['Metric Name']]] = float(row[ix['Metric Value']].replace(',', ''))
        except ValueError:
            pass
        d.setdefault('unit:' + row[ix['Metric Name']], row[ix['Metric Unit']])
    data = list(launches.values())
    sgd = [i for i, d in enumerate(data) if 'fused_sgd' in d['name']]
    step = data[sgd[-2] + 1:sgd[-1] + 1] if len(sgd) >= 2 else data

    def to_ms(d):
        v, u = d.get('gpu__time_duration.sum', 0.0), d.get('unit:gpu__time_duration.sum', 'ns')
        return v * {'ns': 1e-6, 'us': 1e-3, 'ms': 1.0, 's': 1e3}.get(u, 1e-6)

    def to_bytes(d, m):
        v, u = d.get(m, 0.0), d.get('unit:' + m, 'byte')
        return v * {'byte': 1.0, 'Kbyte': 1e3, 'Mbyte': 1e6, 'Gbyte': 1e9}.get(u, 1.0)

    tot, cnt, rd, wr = collections.defaultdict(float), collections.Counter(), collections.defaultdict(float), collections.defaultdict(float)
    for d in step:
        name = d['name'].split('(')[0].replace('void ', '')
        tot[name] += to_ms(d)
        cnt[name] += 1
        rd[name] += to_bytes(d, 'dram__bytes_read.sum')
        wr[name] += to_bytes(d, 'dram__bytes_write.sum')
    total = sum(tot.values())
    have_dram = any(rd.values())
    with open(dst, 'w') as f:
        f.write('# %s\n\n' % title)
        f.write('One training step (ResNet-50, batch 256, 224x224, 1x B200) = the launches between the last two '
                '`fused_sgd` kernels of the ncu launch list (`gpu__time_duration.sum`, `--clock-control none`; '
                'per-launch times are cold-cache and serialised: compare SHARES).\n\n')
        f.write('| kernel | launches | total ms | share |' + (' DRAM read MB | DRAM write MB |' if have_dram else '') + '\n')
        f.write('|---|---:|---:|---:|' + ('---:|---:|' if have_dram else '') + '\n')
        for k, v in sorted(tot.items(), key=lambda kv: -kv[1]):
            f.write('| `%s` | %d | %.3f | %.1f%% |' % (k, cnt[k], v, 100 * v / total))
            f.write(' %.0f | %.0f |\n' % (rd[k] / 1e6, wr[k] / 1e6) if have_dram else '\n')
        f.write('| **sum** | %d | %.3f | 100%% |' % (len(step), total))
        f.write(' %.0f | %.0f |\n' % (sum(rd.values()) / 1e6, sum(wr.values()) / 1e6) if have_dram else '\n')
        ours = sum(v for k, v in tot.items() if k.startswith('b200::'))
        f.write('\nKernels of this repo (`b200::*`): %.1f%% of the step; the rest is torch glue.\n' % (100 * ours / total))
    if js and have_dram:
        out = {}
        for k in tot:
            short = k.replace('b200::', '')
            cls = next((c for p, c in CLASSES.items() if short.startswith(p)), 'other')
            o = out.setdefault(cls, {'launches': 0, 'ms': 0.0, 'dram_read_bytes': 0.0, 'dram_write_bytes': 0.0})
            o['launches'] += cnt[k]; o['ms'] += tot[k]; o['dram_read_bytes'] += rd[k]; o['dram_write_bytes'] += wr[k]
        with open(js, 'w') as f:
            json.dump({'source': src, 'note': 'ncu dram__bytes_read/write.sum summed over the launches of one training step '
                       '(ResNet-50, batch 256, 224x224), grouped by bench.py kernel class', 'classes': out}, f, indent=1)


if __name__ == '__main__':
    main(sys.argv[1], sys.argv[2], sys.argv[3] if len(sys.argv) > 3 else 'ncu launch list summary',
         sys.argv[4] if len(sys.argv) > 4 else None)
