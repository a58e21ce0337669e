#!/bin/bash
# Stages run on the GPU box through gpurun (outputs under gpurun_out/):  bash scripts/gpu.sh <stage> [...]
mkdir -p gpurun_out
for stage in "$@"; do
case $stage in
  step2)      # new kernels, one pytest process per kernel so a device trap in one does not poison the others
    for k in head_prep head_mid similarity_bwd2 addon_bwd2 "bit_reproducible or benchmarked"; do
      n=$(echo $k | tr ' ' '_')
      timeout 600 python -m pytest tests/test_step2_gpu.py -q --tb=short -k "$k" > gpurun_out/t_$n.log 2>&1
      echo "== $k: rc=$? $(tail -1 gpurun_out/t_$n.log)"
    done ;;
  t_*)        # one pytest -k group of tests/test_step2_gpu.py:  t_similarity_bwd2, t_head_mid, ...
    k=${stage#t_}
    timeout 600 python -m pytest tests/test_step2_gpu.py -q --tb=short -k "$k" > gpurun_out/t_$k.log 2>&1
    echo "== $k: rc=$? $(tail -1 gpurun_out/t_$k.log)" ;;
  times64)
    timeout 300 python scripts/step_times.py cub_b64 fp32 > gpurun_out/times_b64.json 2> gpurun_out/times_b64.err; tail -c 1500 gpurun_out/times_b64.json ;;
  timeline)
    timeout 300 python scripts/timeline.py cub_b64 fp32 v2 > gpurun_out/timeline_v2.txt 2> gpurun_out/timeline_v2.err; tail -40 gpurun_out/timeline_v2.txt; tail -3 gpurun_out/timeline_v2.err
    timeout 300 python scripts/timeline.py cub_b64 fp32 v1 > gpurun_out/timeline_v1.txt 2> gpurun_out/timeline_v1.err ;;
  times)
    timeout 300 python scripts/step_times.py cub_b64 fp32 > gpurun_out/times_b64.json 2> gpurun_out/times_b64.err; tail -c 1500 gpurun_out/times_b64.json
    timeout 300 python scripts/step_times.py cub_b64 fp32 1024 > gpurun_out/times_b1024.json 2> gpurun_out/times_b1024.err; tail -c 1500 gpurun_out/times_b1024.json ;;
  sanitize)   # compute-sanitizer memcheck over the small-shape tests of every kernel added in round 2
    timeout 1200 compute-sanitizer --tool memcheck --error-exitcode 9 python -m pytest tests/test_step2_gpu.py tests/test_module_gpu.py \
        tests/test_classmap.py tests/test_gpu_parity.py -q --tb=line -m gpu \
        -k "(tiny or small or cub_b8 or selection_first or dense) and not subprocess and not benchmarked" > gpurun_out/sanitize.log 2>&1
    echo "== sanitize rc=$?"; grep -E "ERROR SUMMARY|Invalid|passed|failed" gpurun_out/sanitize.log | head -20 ;;
  ncu2)       # one --set full capture of each kernel of the five-launch step (second eager step)
    timeout 900 ncu --set full --clock-control none --import-source on -k regex:"head_prep|similarity_tc2|head_mid|sim_grads2|addon_bwd2" \
        -s 5 -c 5 -o gpurun_out/r2_step2 -f python scripts/run_step.py cub_b64 fp32 v2 3 > gpurun_out/ncu2.log 2>&1
    echo "== ncu2 rc=$?"; tail -3 gpurun_out/ncu2.log ;;
  ncuk_*)     # --set full capture of the kernels matching the regex after ncuk_ (five-launch step, second eager step)
    k=${stage#ncuk_}
    timeout 900 ncu --set full --clock-control none --import-source on -k regex:"$k" -s 0 -c 6 -o gpurun_out/r2_$k -f \
        python scripts/run_step.py cub_b64 fp32 v2 3 > gpurun_out/ncuk_$k.log 2>&1
    echo "== ncuk $k rc=$?"; tail -2 gpurun_out/ncuk_$k.log ;;
  ncufinal)   # --set full capture of every kernel of the shipped step (second eager step) -> profiles/r2_ncu_full_step_kernels.txt
    timeout 900 ncu --set full --clock-control none --import-source on \
        -k regex:"select_topk|tcshot|similarity_tc2|head_mid|head_ppc|sim_grads|ppc_rows_add|split_rows" -s 10 -c 10 \
        -o gpurun_out/r2_final -f python scripts/run_step.py cub_b64 fp32 v2 3 > gpurun_out/ncufinal.log 2>&1
    echo "== ncufinal rc=$?"; tail -2 gpurun_out/ncufinal.log ;;
  ncu1)       # same capture of the round-1 launch sequence (reference point for the A/B)
    timeout 900 ncu --set full --clock-control none --import-source on -s 32 -c 16 -o gpurun_out/r2_step1 -f \
        python scripts/run_step.py cub_b64 fp32 v1 3 > gpurun_out/ncu1.log 2>&1
    echo "== ncu1 rc=$?"; tail -3 gpurun_out/ncu1.log ;;
  all)
    timeout 1500 python -m pytest tests -q -m gpu --tb=short > gpurun_out/t_all.log 2>&1; echo "== all: rc=$? $(tail -1 gpurun_out/t_all.log)" ;;
  bench)
    timeout 600 python bench.py > gpurun_out/bench.json 2> gpurun_out/bench.err; tail -c 6000 gpurun_out/bench.json; tail -5 gpurun_out/bench.err ;;
  benchw)     # the other BASELINE configs through --workload
    for w in dogs_b256_eval cars_b64_bf16 "sweep:K=81,D=192,P=2000,B=1024" "sweep:K=196,D=384,P=8000,B=32,eval=1"; do
      n=$(echo $w | tr ':=,' '___')
      timeout 600 python bench.py --workload "$w" --steps 300 --warmup 20 > gpurun_out/bench_$n.json 2> gpurun_out/bench_$n.err
      echo "== $w rc=$?"; tail -c 2500 gpurun_out/bench_$n.json; tail -3 gpurun_out/bench_$n.err
    done ;;
  bench2|bench4|bench8)   # N ranks on one box (gpurun --gpus N): in-graph overlapped all-reduce, then the eager one
    n=${stage#bench}
    timeout 240 python -m torch.distributed.run --nnodes=1 --nproc-per-node $n --master-addr 127.0.0.1 --master-port 29511 \
        bench.py --gpus $n --steps 1000 --warmup 50 --no-extras > gpurun_out/bench_n$n.json 2> gpurun_out/bench_n$n.err
    echo "== in-graph rc=$?"; tail -c 2500 gpurun_out/bench_n$n.json; tail -5 gpurun_out/bench_n$n.err
    timeout 240 python -m torch.distributed.run --nnodes=1 --nproc-per-node $n --master-addr 127.0.0.1 --master-port 29512 \
        bench.py --gpus $n --steps 1000 --warmup 50 --no-extras --exchange nccl > gpurun_out/bench_n${n}_nccl.json 2> gpurun_out/bench_n${n}_nccl.err
    echo "== nccl rc=$?"; tail -c 1200 gpurun_out/bench_n${n}_nccl.json; tail -3 gpurun_out/bench_n${n}_nccl.err ;;
  e2e)
    for e in "" nocopy norows nod2h "nocopy,nosel" "nocopy,nosel,norows"; do EXP=$e timeout 200 python scripts/e2e_timeline.py 32 2 2>&1 | grep "^#"; done
    EXP=nocopy PPH_TIMELINE=1 timeout 200 python scripts/e2e_timeline.py 32 2 2>&1 | grep -v Warn | tail -30 ;;
  tolerances)
    timeout 600 python scripts/measure_tolerances.py > gpurun_out/tolerances.json 2> gpurun_out/tolerances.err; cat gpurun_out/tolerances.json; tail -3 gpurun_out/tolerances.err ;;
  rollout)
    timeout 300 python -m pytest tests/test_rollout_gpu.py -q -m gpu --tb=short 2>&1 | tail -2
    timeout 200 python scripts/rollout_bench.py 2>&1 | cut -c1-150 | tail -4 ;;
  dogscheck)
    timeout 300 python bench.py --workload dogs_b256_eval --steps 200 --warmup 10 --no-extras 2> gpurun_out/dogs.err | python -c "import sys,json; d=json.loads(sys.stdin.read().strip().splitlines()[-1]); print('value %.0f (%.1f us) e2e %.0f'%(d['value'],1e3*d['ms_per_step'],d['e2e']['value']), d['oracle_check'], d['cpu_baseline'] and d['cpu_baseline']['value'])"; tail -2 gpurun_out/dogs.err ;;
  racecheck)  # shared-memory hazard check of the fused selection + add-on forward kernel and the dense PPC kernels (small shapes)
    timeout 170 compute-sanitizer --tool racecheck --error-exitcode 9 python -m pytest tests/test_step2_gpu.py tests/test_module_gpu.py -q --tb=line -m gpu \
        -k "(fused_selection and cub_b8-1-0) or (dense and small)" > gpurun_out/racecheck.log 2>&1
    echo "== racecheck rc=$?"; grep -E "RACECHECK SUMMARY|hazard|passed|failed|Error" gpurun_out/racecheck.log | head -8 ;;
  racecheck2) # the whole default step (cub_b8 fixture) under racecheck: grid-barrier kernels, tcshot epilogues, sparse backward
    timeout 150 compute-sanitizer --tool racecheck --error-exitcode 9 python -m pytest tests/test_step2_gpu.py -q --tb=line -m gpu \
        -k "step_variants and variants1" > gpurun_out/racecheck2.log 2>&1
    echo "== racecheck2 rc=$?"; grep -E "RACECHECK SUMMARY|hazard|passed|failed|Error" gpurun_out/racecheck2.log | head -8 ;;
  execswitch)
    timeout 300 python scripts/exec_switch.py 2>&1 | tail -4 ;;
  gatherparts)
    timeout 200 python scripts/gather_parts.py 2>&1 | tail -5 ;;
  hostgather)
    timeout 200 python scripts/host_gather_times.py 2>&1 | tail -12 ;;
  mgtest)     # multi-GPU pytest group (gpurun --gpus 2)
    timeout 600 python -m pytest tests/test_peer_exchange_multigpu.py -q -m gpu --tb=short > gpurun_out/t_mg.log 2>&1
    echo "== mgtest rc=$? $(tail -1 gpurun_out/t_mg.log)" ;;
  probe2)
    timeout 200 python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29514 \
        scripts/peer_probe.py > gpurun_out/probe2.log 2>&1; echo "== probe2 rc=$?"; grep -v "^W\|^\*\|OMP" gpurun_out/probe2.log | tail -30 ;;
  peer8)      # N = 8, peer exchange only (gpurun --gpus 8)
    timeout 240 python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29551 \
        bench.py --gpus 8 --steps 1000 --warmup 50 --no-extras > gpurun_out/bench_n8.json 2> gpurun_out/bench_n8.err
    echo "== peer8 rc=$?"; tail -c 1500 gpurun_out/bench_n8.json; tail -3 gpurun_out/bench_n8.err ;;
  driver2)    # exactly what the driver runs at N = 2: both arms, default extras, its launch line
    t0=$(date +%s)
    timeout 400 python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29541 \
        bench.py --impl reference --gpus 2 --steps 20 --warmup 3 > gpurun_out/driver2_ref.json 2> gpurun_out/driver2_ref.err
    echo "== reference arm rc=$? $(( $(date +%s) - t0 )) s"; tail -c 700 gpurun_out/driver2_ref.json
    t0=$(date +%s)
    timeout 400 python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29542 \
        bench.py --gpus 2 --steps 500 --warmup 20 > gpurun_out/driver2.json 2> gpurun_out/driver2.err
    echo "== our arm rc=$? $(( $(date +%s) - t0 )) s"; tail -c 1500 gpurun_out/driver2.json; tail -3 gpurun_out/driver2.err ;;
  ddp2|ddp4|ddp8)       # in-graph gradient exchange: result check, step time and kernel timeline at N ranks
    n=${stage#ddp}
    PPH_TIMELINE=1 timeout 200 python -m torch.distributed.run --nnodes=1 --nproc-per-node $n --master-addr 127.0.0.1 --master-port 29513 \
        scripts/ddp_check.py > gpurun_out/ddp$n.log 2>&1; echo "== ddp$n rc=$?"; grep -v "^W\|^\*\|OMP" gpurun_out/ddp$n.log | grep "us/step\|peer_all\|nccl\|next replay" | tail -40 ;;
  smoke)
    timeout 300 python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" 2>&1 | tail -3 ;;
  launches)
    timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none --cache-control none -s 200 -c 60 --csv \
        --log-file gpurun_out/launches.csv python bench.py --steps 20 --warmup 5 --no-cpu --no-extras > gpurun_out/launches.log 2>&1
    echo "== launches rc=$?" ;;
esac
done
