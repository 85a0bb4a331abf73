#!/bin/bash
# One parametrised GPU-box script (replaces the per-round gpu_rNN.sh files): every section writes under gpurun_out/<tag>/.
#   tools/gpu_call.sh <tag> [sections...]     sections: tests tests:<file> smoke bench bench:<workload> refarm ncu_list[:<workload>]
#                                             ncu_full:<workload>:<demangled-name regex> sh:<script> py:<script>
#                                             quick[:<workloads,>]            per-launch times of the steps (no extras), twice each
#                                             kb:<group>                      tools/kbench_c2 (0: c2 launches + per-CTA dump, 1: c3 / c1 shapes)
#                                             multi                           both bench arms under torch.distributed.run on all visible GPUs
#                                             extras                          configs[4] sweep, sanitizer memcheck, step timeline
#                                             exchange                        who publishes the loss sums: loopback A/B of bench.py --exchange
# Every command is bounded by its own timeout (a hung A/B run once cost 25 GPU-minutes).
step_line() { python -c "
import json,sys
d=json.loads(sys.stdin.read()); r=d['roofline']
print('$1 ms_per_step=%.4f stepGBps=%.0f (%.1f%%) | ' % (d['ms_per_step'], r['step_achieved_GBps'], 100*r['step_achieved_GBps']/r['peak']) + ' '.join('%s=%.2fus(%.0f%%)' % (k['part'], k['us'], 100*k['frac']) for k in r['step_kernels']))"; }
quick_bench() { timeout 90 python bench.py --workload $1 --steps 1200 --no-cpu-baseline --no-extras --e2e-steps 3 2>&1 | tail -1; }
tag=${1:-r23}; shift
out=gpurun_out/$tag
mkdir -p $out
for sec in "$@"; do
  case $sec in
    tests)    ( timeout 900 python -m pytest tests -m gpu -q -rfxXs --tb=short 2>&1 | tail -80 ) > $out/pytest_gpu.log; tail -3 $out/pytest_gpu.log ;;
    tests:*)  f=${sec#tests:}; ( timeout 900 python -m pytest $f -m gpu -q -rfxXs -s --tb=short 2>&1 | tail -150 ) > $out/pytest_$(basename $f .py).log; tail -5 $out/pytest_$(basename $f .py).log ;;
    smoke)    ( timeout 200 python -c 'import __graft_entry__ as g; g.smoke()' 2>&1 | tail -3 ) > $out/smoke.log; cat $out/smoke.log ;;
    bench)    ( timeout 600 python bench.py 2>$out/bench.err | tail -1 ) > $out/bench_c2.json; cut -c1-600 $out/bench_c2.json ;;
    bench:*)  w=${sec#bench:}; ( timeout 600 python bench.py --workload $w 2>$out/bench_$w.err | tail -1 ) > $out/bench_$w.json; cut -c1-400 $out/bench_$w.json ;;
    refarm)   ( timeout 600 python bench.py --impl reference 2>$out/bench_ref.err | tail -1 ) > $out/bench_reference.json; cut -c1-400 $out/bench_reference.json ;;
    ncu_list) timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $out/ncu_launches_bench_c2.csv python bench.py --steps 12 --warmup 6 --no-extras --no-cpu-baseline --e2e-steps 3 > $out/ncu_list_bench.log 2>&1; grep -c dct $out/ncu_launches_bench_c2.csv ;;
    ncu_list:*) w=${sec#ncu_list:}; timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 300 --csv --log-file $out/ncu_launches_bench_$w.csv python bench.py --workload $w --steps 8 --warmup 4 --no-extras --no-cpu-baseline --e2e-steps 3 > $out/ncu_list_bench_$w.log 2>&1; grep -c dct $out/ncu_launches_bench_$w.csv ;;
    ncu_full:*) spec=${sec#ncu_full:}; w=${spec%%:*}; k=${spec#*:}; timeout 900 ncu --set full --clock-control none --import-source on --kernel-name-base demangled -k regex:$k -s 6 -c 2 -o $out/ncu_full_${w}_$(echo $k | tr -cd 'A-Za-z0-9_') -f python bench.py --workload $w --steps 8 --warmup 4 --no-extras --no-cpu-baseline --e2e-steps 3 > $out/ncu_full_${w}.log 2>&1; ls -la $out/*.ncu-rep ;;
    quick|quick:*) wls=${sec#quick}; wls=${wls#:}; for wl in $(echo ${wls:-c2,c3,c1,c4} | tr ',' ' '); do for rep in 1 2; do quick_bench $wl | step_line "$wl"; done; done | tee $out/bench_quick.log ;;
    kb:*)     g=${sec#kb:}; [ $g = 0 ] && ( KB_DUMP=1 timeout 100 tools/kbench_c2 200 0 0 2>&1 ) > $out/kbench_c2_dump.log
              ( timeout 200 tools/kbench_c2 200 -1 $g 2>&1 ) > $out/kbench_c2_g$g.log; grep -v "^ " $out/kbench_c2_g$g.log ;;
    multi)    N=$(nvidia-smi -L | wc -l)
              ( timeout 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29517 bench.py --gpus $N --impl reference --steps 3 --warmup 1 2>$out/bench_ref_n$N.err | tail -1 ) > $out/bench_ref_n$N.json; cut -c1-300 $out/bench_ref_n$N.json
              ( timeout 900 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29518 bench.py --gpus $N 2>$out/bench_n$N.err | tail -1 ) > $out/bench_c2_n$N.json; cut -c1-1200 $out/bench_c2_n$N.json
              ( timeout 300 python -m pytest tests/test_gpu_exchange.py -m gpu -q 2>&1 | tail -3 ) ;;
    extras)   ( timeout 300 python tools/sweep.py --no-aten --out $out/sweep 2>&1 | tail -20 ) > $out/sweep.log; cat $out/sweep.log
              ( timeout 600 compute-sanitizer --tool memcheck --error-exitcode 9 python -m pytest tests/test_gpu_parity.py tests/test_gpu_supervised.py -m gpu -q -x -k "consistency_step or ragged or dice or fused or confusion or ce_" 2>&1 | tail -12 ) > $out/sanitizer_memcheck.log; tail -6 $out/sanitizer_memcheck.log
              ( timeout 120 python tools/step_trace.py 2>&1 | tail -8 ) > $out/step_trace_c2.log; cat $out/step_trace_c2.log ;;
    exchange) for rep in 1 2; do for ex in auto p2p p2p-early p2p-fused p2p-deferred; do
                timeout 90 python bench.py --exchange $ex --steps 1200 --no-cpu-baseline --no-extras --e2e-steps 3 2>&1 | tail -1 | python -c "
import json,sys
d=json.loads(sys.stdin.read()); r=d['roofline']
print('c2 exchange=$ex ms_per_step=%.4f launches/step=%d | ' % (d['ms_per_step'], d['gpu_launches']//d['steps']) + ' '.join('%s=%.2fus' % (k['part'], k['us']) for k in r['step_kernels']))"
              done; done | tee $out/ab_exchange_loopback.log ;;
    sh:*)     s=${sec#sh:}; ( timeout 1500 bash $s $out 2>&1 | tail -80 ) > $out/$(basename $s .sh).log; tail -40 $out/$(basename $s .sh).log ;;
    py:*)     s=${sec#py:}; ( timeout 1500 python $s 2>&1 | tail -80 ) > $out/$(basename $s .py).log; tail -40 $out/$(basename $s .py).log ;;
    *) echo "unknown section $sec" ;;
  esac
done
