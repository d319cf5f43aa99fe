#!/bin/bash
# where does the wavefront kernel pay?  frames/s with and without it over a few geometries (MODE_HH + WLS, 28 lanes)
for g in "640,480,64,7" "640,480,128,7" "960,540,128,9" "800,600,64,9" "1280,360,128,9" "512,512,128,9"; do
  a=$(L3D_PROBE_GEOM=$g timeout 120 python tools/skip_probe.py 28 112 2>&1 | tail -1 | sed 's/.*(\(.*\))/\1/')
  b=$(L3D_VWAVE=0 L3D_PROBE_GEOM=$g timeout 120 python tools/skip_probe.py 28 112 2>&1 | tail -1 | sed 's/.*(\(.*\))/\1/')
  echo "$g: wavefront $a   without $b"
done
