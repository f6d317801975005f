set -x
python profiles/tune_stage.py auto 16 > gpurun_out/plain.log 2>&1 && \
ncu --set full --clock-control none --import-source on -k regex:'k_insert_dense|k_scan_dense|k_place_dense|k_pillar_walk' -s 40 -c 4 -o gpurun_out/r02_group_feat python profiles/tune_stage.py auto 16 > gpurun_out/ncu.log 2>&1
tail -3 gpurun_out/ncu.log
