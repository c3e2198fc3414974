#!/bin/bash
# usage: scripts/gpu_run.sh <tag> [what...]   -- runs on the GPU box (through gpurun); outputs under gpurun_out/<tag>_*
tag=$1; shift
what=${*:-"pytest smoke bench"}
mkdir -p gpurun_out
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw --format=csv > gpurun_out/${tag}_smi.txt 2>&1
for w in $what; do
  case $w in
    pytest) timeout 1500 python -m pytest tests -m gpu -q --timeout 900 -x > gpurun_out/${tag}_pytest_gpu.log 2>&1; tail -5 gpurun_out/${tag}_pytest_gpu.log;;
    pytest_all) timeout 1500 python -m pytest tests -m gpu -q --timeout 900 > gpurun_out/${tag}_pytest_gpu.log 2>&1; tail -15 gpurun_out/${tag}_pytest_gpu.log;;
    smoke) timeout 600 python -c "import __graft_entry__ as g; g.smoke()" > gpurun_out/${tag}_smoke.log 2>&1; tail -3 gpurun_out/${tag}_smoke.log;;
    bench) timeout 900 python bench.py --steps 10 --warmup 3 --layers gpurun_out/${tag}_layers.txt > gpurun_out/${tag}_bench.json 2> gpurun_out/${tag}_bench.err; tail -c 600 gpurun_out/${tag}_bench.json; tail -3 gpurun_out/${tag}_bench.err;;
    bench_kitti|bench_fov180|bench_fov108|bench_oxford)
      declare -A m=([bench_kitti]=kitti_b32 [bench_fov180]=vigor_prior72_fov180 [bench_fov108]=vigor_prior72_fov108 [bench_oxford]=oxford_b1)
      k=${m[$w]}
      timeout 900 python bench.py --workload $k --steps 10 --warmup 3 --layers gpurun_out/${tag}_layers_$k.txt > gpurun_out/${tag}_bench_$k.json 2> gpurun_out/${tag}_bench_$k.err; head -c 400 gpurun_out/${tag}_bench_$k.json; echo; tail -3 gpurun_out/${tag}_bench_$k.err;;
    pytest_match) timeout 900 python -m pytest tests/test_gpu_kernels.py -m gpu -q --timeout 600 -k match > gpurun_out/${tag}_pytest_match.log 2>&1; tail -8 gpurun_out/${tag}_pytest_match.log;;
    pytest_train) timeout 1200 python -m pytest tests/test_gpu_train.py -m gpu -q --timeout 900 > gpurun_out/${tag}_pytest_train.log 2>&1; tail -25 gpurun_out/${tag}_pytest_train.log;;
    bench_train) timeout 900 python bench.py --workload train --steps 5 --warmup 3 --layers gpurun_out/${tag}_layers_train.txt > gpurun_out/${tag}_bench_train.json 2> gpurun_out/${tag}_bench_train.err; head -c 700 gpurun_out/${tag}_bench_train.json; echo; tail -5 gpurun_out/${tag}_bench_train.err;;
    bench_train_fp32) timeout 900 python bench.py --workload train --precision fp32 --steps 3 --warmup 3 --no-cpu --layers gpurun_out/${tag}_layers_train_fp32.txt > gpurun_out/${tag}_bench_train_fp32.json 2> gpurun_out/${tag}_bench_train_fp32.err; head -c 500 gpurun_out/${tag}_bench_train_fp32.json; echo; tail -5 gpurun_out/${tag}_bench_train_fp32.err;;
    profile_train) timeout 600 python scripts/profile_train.py > gpurun_out/${tag}_profile_train.txt 2>&1; head -40 gpurun_out/${tag}_profile_train.txt | cut -c1-200;;
    bench_dw) timeout 300 python scripts/bench_dwconv.py fast > gpurun_out/${tag}_bench_dw.txt 2>&1; tail -2 gpurun_out/${tag}_bench_dw.txt;;
    ncu_igemm_halo) timeout 600 ncu --set full --clock-control none --import-source on -k regex:igemm_tcgen05 -s 6 -c 1 -o gpurun_out/${tag}_prof_igemm_halo python scripts/bench_igemm.py conv 16 160 40 160 64 > gpurun_out/${tag}_ncu_igemm_halo.log 2>&1; tail -3 gpurun_out/${tag}_ncu_igemm_halo.log | cut -c1-200;;
    ncu_ring2b) timeout 600 ncu --set full --clock-control none --import-source on -k regex:conv_ring -s 6 -c 1 -o gpurun_out/${tag}_prof_ring2b python scripts/bench_igemm.py conv 16 40 0 40 256 > gpurun_out/${tag}_ncu_ring2b.log 2>&1; tail -3 gpurun_out/${tag}_ncu_ring2b.log | cut -c1-200;;
    bench_ring) for a in "16 40 0 40 256" "16 40 16 40 256" "16 32 16 32 256" "16 32 0 32 256" "16 16 0 16 512" "16 80 24 80 128" "16 80 0 80 128"; do timeout 120 python scripts/bench_igemm.py conv $a 2>&1 | tail -1; done | tee gpurun_out/${tag}_bench_ring.txt;;
    test_conv) timeout 600 python -m pytest tests/test_gpu_kernels.py -m gpu -q -k "conv3x3 or deconv or k2s2" 2>&1 | tail -4;;
    test_dw) timeout 600 python -m pytest tests/test_gpu_kernels.py tests/test_fast_encoder.py -m gpu -q -k "dwconv or encoder" 2>&1 | tail -4;;
    probe2) timeout 120 scripts/tma_probe2.bin 2>&1 | tee gpurun_out/${tag}_tma_probe2.txt;;
    test_proj) timeout 600 python -m pytest tests/test_gpu_kernels.py tests/test_fast_encoder.py tests/test_gpu_forward.py -m gpu -q -x -k "mbconv_project or encoder or bit_reproducible or bf16" 2>&1 | tail -6;;
    ncu_dwtile) timeout 600 ncu --set full --clock-control none --import-source on -k regex:dwconv_tile -s 2 -c 1 -o gpurun_out/${tag}_prof_dwtile python scripts/prof_dwconv.py > gpurun_out/${tag}_ncu_dwtile.log 2>&1; tail -3 gpurun_out/${tag}_ncu_dwtile.log | cut -c1-200;;
    launches) CCVPE_NCU_RANGE=1 timeout 900 ncu --profile-from-start off --metrics gpu__time_duration.sum --clock-control none -c 800 --csv --log-file gpurun_out/${tag}_launches.csv python bench.py --steps 1 --warmup 3 --no-cpu --no-parity --no-torch-gpu-baseline > gpurun_out/${tag}_ncu_bench.log 2>&1; python scripts/launch_shares.py gpurun_out/${tag}_launches.csv | tee gpurun_out/${tag}_launch_shares.txt | head -32;;
    bench_pw) timeout 300 python scripts/bench_pointwise.py 64 2>&1 | tee gpurun_out/${tag}_bench_pw.txt | tail -26;;
    ncu_pw) timeout 600 ncu --set full --clock-control none --import-source on -k regex:igemm_tcgen05 -s 2 -c 1 -o gpurun_out/${tag}_prof_pw python scripts/bench_pointwise.py 64 0 > gpurun_out/${tag}_ncu_pw.log 2>&1; tail -3 gpurun_out/${tag}_ncu_pw.log | cut -c1-200;;
    test_enc) timeout 900 python -m pytest tests/test_gpu_kernels.py tests/test_fast_encoder.py tests/test_gpu_forward.py -m gpu -q -x -k "mbconv_project or se_gate or conv3x3 or deconv or encoder or bit_reproducible or bf16" 2>&1 | tail -6;;
    test_stem) timeout 900 python -m pytest tests/test_gpu_kernels.py tests/test_fast_encoder.py tests/test_gpu_forward.py -m gpu -q -x -k "stem or encoder or bit_reproducible or bf16 or uint8" 2>&1 | tail -6;;
    bench_enc_ops) for a in "project 64 12800 144 24 1" "project 64 51200 32 16 0" "project 64 200 1152 192 1" "project 64 800 480 80 1" "stem 64 512 512 0 0" "stem 64 320 640 1 0" "stem 64 512 512 0 1"; do timeout 120 python scripts/bench_encoder_ops.py $a 2>&1 | tail -1; done | tee gpurun_out/${tag}_bench_enc_ops.txt;;
    ncu_stem) timeout 600 ncu --set full --clock-control none --import-source on -k regex:stem_tcgen05 -s 4 -c 1 -o gpurun_out/${tag}_prof_stem python scripts/bench_encoder_ops.py stem 64 512 512 0 0 > gpurun_out/${tag}_ncu_stem.log 2>&1; tail -2 gpurun_out/${tag}_ncu_stem.log | cut -c1-200;;
    ncu_project) timeout 600 ncu --set full --clock-control none --import-source on -k regex:project_tcgen05 -s 4 -c 1 -o gpurun_out/${tag}_prof_project python scripts/bench_encoder_ops.py project 64 12800 144 24 1 > gpurun_out/${tag}_ncu_project.log 2>&1; tail -2 gpurun_out/${tag}_ncu_project.log | cut -c1-200;;
    ncu_halo3) timeout 600 ncu --set full --clock-control none --import-source on -k regex:igemm_tcgen05 -s 6 -c 1 -o gpurun_out/${tag}_prof_igemm_halo3 python scripts/bench_igemm.py conv 16 80 24 80 128 > gpurun_out/${tag}_ncu_halo3.log 2>&1; tail -2 gpurun_out/${tag}_ncu_halo3.log | cut -c1-200;;
    ncu_match1) timeout 600 ncu --set full --clock-control none --import-source on -k regex:match_tcgen05 -s 4 -c 1 -o gpurun_out/${tag}_prof_match1 python scripts/bench_match.py 64 1280 8 20 64 tc > gpurun_out/${tag}_ncu_match1.log 2>&1; tail -2 gpurun_out/${tag}_ncu_match1.log | cut -c1-200; timeout 120 python scripts/bench_match.py 64 1280 8 20 64 tc | tail -1; timeout 120 python scripts/bench_match.py 1 1280 8 20 64 tc | tail -1;;
    *) echo "unknown step $w";;
  esac
done
