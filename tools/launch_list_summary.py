"""Summarises an ncu launch list (CSV of gpu__time_duration.sum, dram__bytes_read.sum, dram__bytes_write.sum per
launch, as written by tools/gpu/launch_list.sh) into the per-kernel / per-family markdown table under profiles/.

  python tools/launch_list_summary.py gpurun_out/launches.csv profiles/rNN_step_launches.md "title" ["note"]
"""
import collections
import csv
import json
import re
import sys

FAMILIES = [
    ('conv', r'k_igemm|k_halo3x3|k_stem_s2d|k_splitk|k_im2col|k_simt|k_pack_weights|k_s2d'),
    ('bn', r'k_bn_'),
    ('pool', r'k_maxpool'),
    ('optimizer', r'k_sgd|multi_tensor_apply'),
    ('mask update', r'k_hist_drop|k_pick_drop|k_scan_|k_resolve|k_publish|k_noise'),
    ('mask ops', r'k_apply_mask|k_popcount|k_pack_f32|k_unpack'),
]


def main():
  src, out, title = sys.argv[1:4]
  note = sys.argv[4] if len(sys.argv) > 4 else ''
  rows = list(csv.reader(open(src)))
  start = [i for i, r in enumerate(rows) if r and r[0] == 'ID'][0]
  hdr = rows[start]
  col = {h: i for i, h in enumerate(hdr)}
  per = collections.OrderedDict()
  launches = {}
  for r in rows[start + 1:]:
    if len(r) < len(hdr):
      continue
    name = re.sub(r'^(void )?(rigl::)?', '', r[col['Kernel Name']])
    name = re.sub(r'\(.*$', '', name)[:72]
    metric, unit, val = r[col['Metric Name']], r[col['Metric Unit']], float(r[col['Metric Value']].replace(',', ''))
    d = per.setdefault(name, collections.Counter())
    if metric == 'gpu__time_duration.sum':
      val *= {'ns': 1e-6, 'us': 1e-3, 'ms': 1.0, 'nsecond': 1e-6, 'usecond': 1e-3, 'msecond': 1.0}.get(unit, 1e-6)
      d['ms'] += val
      d['n'] += 1
    else:
      val *= {'byte': 1, 'Kbyte': 1e3, 'Mbyte': 1e6, 'Gbyte': 1e9}.get(unit, 1)
      d['rd' if 'read' in metric else 'wr'] += val
  total = sum(d['ms'] for d in per.values())
  n_total = sum(d['n'] for d in per.values())
  lines = ['# ' + title, '']
  if note:
    lines += [note, '']
  lines += ['Per-launch times under ncu are cold-cache (ncu flushes caches before every kernel, so producer -> consumer '
            'reuse through L2 shows up as DRAM traffic) and serialised: compare SHARES; DRAM bytes are per step.', '',
            'launches: %d, summed kernel time: %.3f ms' % (n_total, total), '',
            '| kernel | launches | ms | share | DRAM rd GB | DRAM wr GB |', '|---|---|---|---|---|---|']
  for name, d in sorted(per.items(), key=lambda kv: -kv[1]['ms']):
    lines.append('| `%s` | %d | %.3f | %.1f%% | %.2f | %.2f |' % (name, d['n'], d['ms'], 100 * d['ms'] / total,
                                                                 d['rd'] / 1e9, d['wr'] / 1e9))
  fam_json = {}
  for fam, pat in FAMILIES:
    sel = [d for n, d in per.items() if re.search(pat, n)]
    if not sel:
      continue
    ms, n = sum(d['ms'] for d in sel), sum(d['n'] for d in sel)
    gb = sum(d['rd'] + d['wr'] for d in sel) / 1e9
    lines += ['', '%s family: %d launches, %.3f ms (%.1f%%), %.2f GB DRAM traffic' % (fam, n, ms, 100 * ms / total, gb)]
    fam_json[fam] = {'launches': n, 'ms': ms, 'dram_bytes': gb * 1e9}
  open(out, 'w').write('\n'.join(lines) + '\n')
  if 'conv' in fam_json:
    jpath = re.sub(r'step_launches.*\.md$', 'dram_traffic_step.json', out)
    if jpath != out:
      json.dump({'conv_family_dram_bytes_per_step': fam_json['conv']['dram_bytes'],
                 'conv_family_launches': fam_json['conv']['launches'], 'families': fam_json, 'source': src,
                 'command': 'ncu --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum '
                            '--clock-control none --profile-from-start off python tools/step_for_ncu.py --steps 1 --warmup 2'},
                open(jpath, 'w'), indent=1)
  print('\n'.join(lines[:60]))


if __name__ == '__main__':
  main()
