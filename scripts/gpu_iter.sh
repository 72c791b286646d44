# one measurement iteration on the B200 box: GPU parity tests, short bench (2 h of audio), one ncu --set full capture
mkdir -p gpurun_out
python -m pytest tests -m gpu -x -q 2>&1 | tail -4
python bench.py --hours ${HOURS:-2} --steps 3 --warmup 3 --no-e2e --no-cpu --no-weak 2>&1 | python -c "
import sys, json
for ln in sys.stdin:
    ln=ln.strip()
    if ln.startswith('{'):
        d=json.loads(ln); r=d['roofline']
        print('ms/step %.2f  frame %.2f  finalize %.2f  value %.0f  frac %.4f launches %d clocks %s' % (d['ms_per_step'], r['kernel_ms_per_step'], r['finalize_ms_per_step'], d['value'], r['frac'], d['gpu_launches'], d['clocks']))
    else: print(ln)
"
if [ -n "$NAME" ]; then
  CMD="python bench.py --hours 0.5 --steps 1 --warmup 1 --no-e2e --no-cpu --no-weak"
  $CMD > gpurun_out/ncu_plain.log 2>&1 && ncu --set full --clock-control none --import-source on -k regex:${KERNEL:-frame_warp} -s ${SKIP:-4} -c 1 -f -o gpurun_out/$NAME $CMD > gpurun_out/ncu_run.log 2>&1
  tail -2 gpurun_out/ncu_run.log
fi
