#!/bin/bash
# A/B of a runtime switch: scene throughput with and without `VAR=VALUE` (e.g. tools/ab_env.sh RT1W_TAIL_FACTOR=4 "stress:8 final_scene:32")
SW=${1:-RT1W_FACE_GROUPS=0}; SCENES=${2:-cornel_box:100}
for env in "RT1W_NOOP=1" "$SW"; do
  echo "== $env"
  for i in 1 2; do
  env $env timeout 600 python tools/scene_perf.py $SCENES 2>/dev/null | python -c "
import sys,json
for l in sys.stdin:
    if l.startswith('{'):
        d=json.loads(l); print(' ', d['scene'], d['image'], 'spp', d['spp'], 'ms', d['render_ms'], 'Mpaths/s', d['mpaths_s'], 'Mrays/s', d['mrays_s'], 'rays/path', d['rays_per_path'])"
  done
done
