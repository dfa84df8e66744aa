# forward kernel A/B in one call: smplpp_b200/lib_<name>.so for each name given (default: old new old new), in order
run() {
  timeout 300 python bench.py --steps 20 --warmup 5 --no-cpu-baseline --no-ik | python -c "
import json,sys; d=json.loads(sys.stdin.read()); r=d['roofline']; l=r['lbs']; e=d['e2e']
print('value %.3f M  ms/launch %.4f  burst %.4f  frac %.3f  diff %.2e' % (d['value']/1e6, r['ms_per_launch'], r['burst_ms_per_launch'], r['frac'], e['max_abs_diff_vs_device_path']))
print('  lbs ms/launch %.4f  4x4 %.4f  other variants %s' % (l['ms_per_launch'], l['ms_per_launch_4x4_transforms'], '  '.join('%s %.4f' % kv for kv in sorted(l['ms_per_launch_other_variants'].items()))))
print('  e2e %.3f M meshes/s  pageable %.3f M  d2h %.1f GB/s' % (e['value']/1e6, e['pageable_value']/1e6, e['d2h_gbs']))"
}
for v in ${*:-old new old new}; do
  cp smplpp_b200/lib_$v.so smplpp_b200/libsmplpp_b200.so
  echo "== $v"; run
done
