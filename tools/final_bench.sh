#!/bin/bash
# Round-2 measurement set, as committed under profiles/ (run on a B200 box through gpurun; ~14 GPU-minutes):
#   bench lines (ours + the CPU reference arm), ncu launch list of the bench command, ncu --set full of the data-flow
#   kernel (16 frames) and of the tcgen05 kernel (bs=256, 8 frames), DRAM traffic of the bench's own 1024-frame launch and of
#   a bs=256 launch, phase tables, the data-flow kernel's cycle / skew trace and the team timings.
set -u
O=gpurun_out
T=${1:-r2z}
python bench.py --impl reference --steps 3 --warmup 1 > $O/${T}_bench_reference.json 2> $O/${T}_bench_reference.err
python bench.py > $O/${T}_bench.json 2> $O/${T}_bench.err
# launch list of the same command (short form): per-launch times are cold-cache and serialised, the SHARE must agree
CMD="python bench.py --steps 2 --warmup 3 --configs none --no-cpu-baseline"
$CMD > $O/${T}_plain_list.log 2>&1 && ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $O/${T}_launches_bench.csv $CMD > $O/${T}_ncu_list.log 2>&1
# data-flow kernel: full set on a 16-frame launch; DRAM bytes of one 1024-frame launch at the bench's context
python tools/ll_ncu.py --frames 16 > $O/${T}_ll_plain.log 2>&1 && ncu --set full --clock-control none --import-source on -k regex:smol_ll2_kernel -s 1 -c 1 -o $O/${T}_ll2 python tools/ll_ncu.py --frames 16 > $O/${T}_ll_ncu.log 2>&1
ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum --clock-control none -k regex:smol_ll2_kernel -s 1 -c 1 --csv --log-file $O/${T}_ll2_traffic_1024.csv python tools/ll_ncu.py --frames 1024 > $O/${T}_ll_traffic.log 2>&1
# tcgen05 kernel at bs=256: full set on an 8-frame launch (the decode launch after prefill + warm-up), DRAM bytes
TC="python bench.py --batch 256 --frames 8 --prompt-bytes 64 --steps 1 --warmup 3 --configs none --no-cpu-baseline"
$TC > $O/${T}_tc_plain.log 2>&1 && ncu --set full --clock-control none --import-source on -k regex:smol_decode_kernel -s 6 -c 2 -o $O/${T}_tc $TC > $O/${T}_tc_ncu.log 2>&1
ncu --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum --clock-control none -k regex:smol_decode_kernel -c 12 --csv --log-file $O/${T}_launches_bs256.csv $TC > $O/${T}_tc_list.log 2>&1
timeout 300 python tools/phase_profile.py --batch 256 --frames 16 --prompt-bytes 64 > $O/${T}_phase_bs256.log 2>&1
timeout 300 python tools/phase_profile.py --batch 256 --frames 16 --prompt-bytes 400 > $O/${T}_phase_bs256_L420.log 2>&1
timeout 300 python tools/phase_profile.py --batch 64 --frames 16 --sampled > $O/${T}_phase_bs64_sampled.log 2>&1
timeout 400 python tools/ll2_probe.py --skip-check --holdoffs 400 > $O/${T}_probe.log 2>&1
timeout 400 python tools/ll2_probe.py --skip-check --skip-timing --teams > $O/${T}_teams.log 2>&1
# Mimi streaming decoder (the step after the path): step times, launch lists, DRAM bytes of a step, ncu of the row / tile kernels,
# streaming and serving through both engines
timeout 300 python tools/mimi_bench.py --batch 1,4,8,16,32,64 > $O/${T}_mimi_steps.log 2>&1
timeout 400 python tools/mimi_bench.py --batch 1 --frames 1024 >> $O/${T}_mimi_steps.log 2>&1
for B in 1 64; do
  ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum --clock-control none -c 600 --csv --log-file $O/${T}_mimi_traffic_bs$B.csv python tools/mimi_bench.py --batch $B --frames 4 --mode eager > /dev/null 2>&1
done
ncu --set full --cache-control none --clock-control none --import-source on -k regex:tile_kernel -s 30 -c 3 -o $O/${T}_mimi_tile python tools/mimi_bench.py --batch 64 --frames 4 --mode eager > /dev/null 2>&1
ncu --set full --cache-control none --clock-control none --import-source on -k regex:lin_kernel -s 60 -c 4 -o $O/${T}_mimi_lin python tools/mimi_bench.py --batch 1 --frames 4 --mode eager > /dev/null 2>&1
timeout 400 python bench.py --configs tts_stream_bs1 --steps 2 --warmup 3 --no-cpu-baseline > $O/${T}_tts_stream.json 2>/dev/null
timeout 400 python bench.py --configs tts_stream_bs1 --steps 2 --warmup 3 --no-cpu-baseline --no-stream-overlap > $O/${T}_tts_stream_plain.json 2>/dev/null
timeout 600 python tools/tts_serving_bench.py > $O/${T}_tts_serving.log 2>&1
python -c "import __graft_entry__ as g; g.smoke()" > $O/${T}_smoke.log 2>&1
tail -3 $O/${T}_bench.json | cut -c1-600
