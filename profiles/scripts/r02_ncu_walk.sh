python profiles/tune_stage.py auto 16 > gpurun_out/plain.log 2>&1 && \
ncu --set full --clock-control none --import-source on -k regex:'k_pillar_walk' -s 10 -c 1 -o gpurun_out/r02_walk python profiles/tune_stage.py auto 16 > gpurun_out/ncu.log 2>&1
tail -2 gpurun_out/ncu.log; cat gpurun_out/plain.log
