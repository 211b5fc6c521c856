#!/bin/bash
# Round-end rehearsal on one GPU + the captures behind profiles/<TAG>_*: smoke, the GPU tests, both bench arms as the driver runs
# them, the launch list of the bench command, one `ncu --set full` capture of a steady-state wave per BASELINE config, and
# ncu-counted flops of one whole render per config, digested on the box by tools/profiles_refresh.sh into
# gpurun_out/profiles_<TAG>/ (summaries, regions, metrics, <TAG>_flops.json).  Afterwards, here:
#     copy the files of profiles_<TAG>/ into profiles/
#     gpurun --timeout 2400 -- 'bash tools/profiles_capture.sh r02'
TAG=${1:-r02}
mkdir -p gpurun_out
if [ -z "${2:-}" ]; then
python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -1
python -m pytest tests -m gpu -q --tb=short 2>&1 | tail -3
python bench.py --impl reference > gpurun_out/${TAG}_bench_reference.json 2> gpurun_out/${TAG}_bench_reference.err
python bench.py > gpurun_out/${TAG}_bench.json 2> gpurun_out/${TAG}_bench.err || tail -5 gpurun_out/${TAG}_bench.err
CMD="python bench.py --steps 1 --warmup 1 --no-cpu-baseline --no-configs"
ncu --metrics gpu__time_duration.sum --clock-control none -c 700 --csv --log-file gpurun_out/${TAG}_launches.csv $CMD > gpurun_out/${TAG}_ncu_launches.log 2>&1
fi
M=smsp__sass_thread_inst_executed_op_fadd_pred_on.sum,smsp__sass_thread_inst_executed_op_fmul_pred_on.sum,smsp__sass_thread_inst_executed_op_ffma_pred_on.sum,smsp__sass_thread_inst_executed_op_dadd_pred_on.sum,smsp__sass_thread_inst_executed_op_dmul_pred_on.sum,smsp__sass_thread_inst_executed_op_dfma_pred_on.sum,smsp__thread_inst_executed.sum
export RT1W_NO_WARMUP=1
ONLY=${2:-} # optional: capture these configs only (e.g. "C2 C3"), skipping smoke / tests / bench lines
for spec in C1:cornel_box:100:3 C2:random_scene:32:2:1200 C2w:one_weekend:32:2 C3:final_scene:32:2 C5:stress:8:1; do
  IFS=: read name scene spp skip width <<< "$spec"
  [ -n "$ONLY" ] && ! echo " $ONLY " | grep -q " $name " && continue
  [ -n "$width" ] && spp=$spp:$width # the config's own image size (random_scene defaults to the reference's 400 x 225)
  timeout 900 ncu --set full --clock-control none --import-source on -k regex:k_wave -s $skip -c 1 -f -o gpurun_out/${TAG}_${name}_wave python tools/scene_perf.py $scene:$spp > gpurun_out/${TAG}_${name}_full.log 2>&1
  timeout 900 ncu --metrics $M --clock-control none -k regex:k_wave -c 400 --csv --log-file gpurun_out/${TAG}_${name}_flops.csv python tools/scene_perf.py $scene:$spp > gpurun_out/${TAG}_${name}_flops.json 2> gpurun_out/${TAG}_${name}_flops.err
done
# digest here (the .ncu-rep files are ~10 MB each: more than gpurun brings back), then drop them
bash tools/profiles_refresh.sh ${TAG} gpurun_out/profiles_${TAG} > /dev/null 2>&1
rm -f gpurun_out/${TAG}_*_wave.ncu-rep gpurun_out/${TAG}_*_flops.csv
ls -la gpurun_out/profiles_${TAG} | head -40
