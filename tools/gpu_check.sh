#!/bin/bash
# One GPU-box call: smoke + the -m gpu suite + a short bench + the host/PCIe topology, everything into gpurun_out/.
#   gpurun --timeout 1500 -- 'bash tools/gpu_check.sh [tests|bench|topo|all] [extra bench args]'
# Multi-GPU: gpurun --gpus N -- 'bash tools/gpu_check.sh benchN N'
set -u
mkdir -p gpurun_out
what=${1:-all}
shift || true
topo() {
  { echo "== nvidia-smi topo -m"; nvidia-smi topo -m; echo "== nvidia-smi -L"; nvidia-smi -L;
    echo "== lscpu"; lscpu | head -30; echo "== numa nodes"; ls /sys/devices/system/node/ 2>/dev/null; cat /sys/devices/system/node/node*/cpulist 2>/dev/null;
    echo "== meminfo"; head -5 /proc/meminfo; echo "== nproc"; nproc;
    echo "== pci"; for d in /sys/bus/pci/devices/*; do c=$(cat $d/class 2>/dev/null); case $c in 0x0302*|0x0300*) echo "$d class=$c numa=$(cat $d/numa_node) local_cpulist=$(cat $d/local_cpulist) link=$(cat $d/current_link_speed 2>/dev/null) x$(cat $d/current_link_width 2>/dev/null)";; esac; done;
    echo "== lspci -tv"; lspci -tv 2>/dev/null | head -80; } > gpurun_out/topology.txt 2>&1
}
case $what in
  tests|all)
    timeout 120 python __graft_entry__.py --smoke > gpurun_out/smoke.log 2>&1; echo "smoke rc=$?"
    timeout 1200 python -m pytest tests -m gpu -x -q > gpurun_out/pytest_gpu.log 2>&1; echo "pytest rc=$?"; tail -5 gpurun_out/pytest_gpu.log
    ;;&
  bench|all)
    timeout 900 python bench.py --steps 20 --warmup 5 "$@" > gpurun_out/bench_n1.json 2> gpurun_out/bench_n1.err; echo "bench rc=$?"; tail -3 gpurun_out/bench_n1.err
    head -c 1500 gpurun_out/bench_n1.json
    ;;&
  topo|all)
    topo
    ;;
  utf8)
    # Utf8 columns: dictionary-encoding throughput and string queries vs the same queries over a UInt32 column
    # -> profiles/r03_utf8_<rows>.json (the same JSON lines are printed as they are measured)
    timeout 1200 python tools/bench_utf8.py "$@"; echo "bench_utf8 rc=$?"
    ;;
  select)
    # select-kernel shapes: timings with the dense build available (tma) / never launched (sparse), then ncu --set full of the dense / third / 1-in-1024 selections
    for v in tma sparse; do FQ_SEL_VARIANT=$v timeout 600 python tools/bench_select.py 2>&1; echo "$v rc=$?"; done
    for c in all third 1024; do
      timeout 600 ncu --set full --clock-control none --import-source on -k regex:select --launch-skip 2 --launch-count 1 -o gpurun_out/ncu_select_$c -f python tools/prof_select.py 1000000000 $c > gpurun_out/ncu_select_$c.log 2>&1; echo "ncu $c rc=$?"
    done
    ;;
  recapture)
    # the captures that changed after the main `profiles` pass: final GROUP BY kernels, validity bitmaps staged through the ring
    cap() { name=$1; regex=$2; shift 2; timeout 600 ncu --set full --clock-control none --import-source on -k regex:$regex --launch-skip 2 --launch-count 1 -o gpurun_out/ncu_$name -f "$@" > gpurun_out/ncu_$name.log 2>&1; echo "ncu $name rc=$?";
            ncu -i gpurun_out/ncu_$name.ncu-rep --page details > gpurun_out/ncu_$name.details.txt 2>/dev/null;
            ncu -i gpurun_out/ncu_$name.ncu-rep --page raw --csv > gpurun_out/ncu_$name.raw.csv 2>/dev/null; rm -f gpurun_out/ncu_$name.ncu-rep; }
    cap agg_nullable_bits_1e9 "_agg_" python tools/prof_agg.py 1000000000 nullable_bits
    cap agg_nullable_u8_bits_4e9 "_agg_" python tools/prof_agg.py 4000000000 nullable_u8_bits
    for k in 7 1000 5000 1000000; do cap groupby_k${k}_1e9 groupby python tools/prof_groupby.py 1000000000 $k; done
    ;;
  sortcap)
    # ORDER BY kernels: the scatter and the histogram of one pass over 2.5e8 scrambled 64-bit keys
    cap() { name=$1; regex=$2; shift 2; timeout 600 ncu --set full --clock-control none --import-source on -k regex:$regex --launch-skip 3 --launch-count 1 -o gpurun_out/ncu_$name -f "$@" > gpurun_out/ncu_$name.log 2>&1; echo "ncu $name rc=$?";
            ncu -i gpurun_out/ncu_$name.ncu-rep --page details > gpurun_out/ncu_$name.details.txt 2>/dev/null;
            ncu -i gpurun_out/ncu_$name.ncu-rep --page raw --csv > gpurun_out/ncu_$name.raw.csv 2>/dev/null; rm -f gpurun_out/ncu_$name.ncu-rep; }
    cap sort_scatter_2.5e8 fq_sort_scatter python tools/prof_sort.py 250000000 scrambled
    cap sort_hist_2.5e8 fq_sort_hist python tools/prof_sort.py 250000000 scrambled
    ;;
  profiles)
    # ncu captures for profiles/: every kernel of the path, --set full, one launch each after warm-up
    # (the .ncu-rep files are summarised on the box and removed: gpurun copies back at most 64 MiB)
    cap() { name=$1; regex=$2; shift 2; timeout 600 ncu --set full --clock-control none --import-source on -k regex:$regex --launch-skip 2 --launch-count 1 -o gpurun_out/ncu_$name -f "$@" > gpurun_out/ncu_$name.log 2>&1; echo "ncu $name rc=$?";
            ncu -i gpurun_out/ncu_$name.ncu-rep --page details > gpurun_out/ncu_$name.details.txt 2>/dev/null;
            ncu -i gpurun_out/ncu_$name.ncu-rep --page raw --csv > gpurun_out/ncu_$name.raw.csv 2>/dev/null;
            case $name in agg_headline_1e10|select_all_1e9) ;; *) rm -f gpurun_out/ncu_$name.ncu-rep;; esac; }
    rm -f gpurun_out/*.ncu-rep
    cap agg_headline_1e10 agg_tma python tools/prof_agg.py 10000000000 headline
    cap agg_headline_gen_1e10 "_agg_" python tools/prof_agg.py 10000000000 headline gen
    cap agg_nullable_bytes_1e9 "_agg_" python tools/prof_agg.py 1000000000 nullable
    cap agg_nullable_bits_1e9 "_agg_" python tools/prof_agg.py 1000000000 nullable_bits
    cap agg_nullable_u8_bytes_4e9 "_agg_" python tools/prof_agg.py 4000000000 nullable_u8
    cap agg_nullable_u8_bits_4e9 "_agg_" python tools/prof_agg.py 4000000000 nullable_u8_bits
    cap select_readme_1e9 select_tma python tools/prof_select.py 1000000000 readme
    cap select_all_1e9 select_dense python tools/prof_select.py 1000000000 all
    cap select_third_1e9 select_dense python tools/prof_select.py 1000000000 third
    cap select_1024_1e9 select_tma python tools/prof_select.py 1000000000 1024
    cap map_1e9 map_tma python tools/prof_select.py 1000000000 map
    timeout 600 ncu --set full --clock-control none -k regex:fq_fill_numbers --launch-count 1 -o gpurun_out/ncu_fill_1e9 -f python tools/prof_select.py 1000000000 map > gpurun_out/ncu_fill_1e9.log 2>&1; echo "ncu fill rc=$?"
    ncu -i gpurun_out/ncu_fill_1e9.ncu-rep --page details > gpurun_out/ncu_fill_1e9.details.txt 2>/dev/null; ncu -i gpurun_out/ncu_fill_1e9.ncu-rep --page raw --csv > gpurun_out/ncu_fill_1e9.raw.csv 2>/dev/null; rm -f gpurun_out/ncu_fill_1e9.ncu-rep
    cap groupby_k7_1e9 groupby python tools/prof_groupby.py 1000000000 7
    cap groupby_k1000_1e9 groupby python tools/prof_groupby.py 1000000000 1000
    cap groupby_k1e6_1e9 groupby python tools/prof_groupby.py 1000000000 1000000
    timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file gpurun_out/launches_bench.csv python bench.py --steps 20 --warmup 5 --no-cpu-baseline --no-query-table --e2e-rows 1000000000 > gpurun_out/launches_bench.log 2>&1; echo "launch list rc=$?"
    ;;
  benchN)
    N=$1; shift
    topo
    timeout 900 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29511 bench.py --gpus $N --steps 20 --warmup 5 "$@" > gpurun_out/bench_n$N.json 2> gpurun_out/bench_n$N.err; echo "bench N=$N rc=$?"; tail -5 gpurun_out/bench_n$N.err
    head -c 1500 gpurun_out/bench_n$N.json
    ;;
esac
