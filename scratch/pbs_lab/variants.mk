VARIANTS := r1 final ws2
R1 := -DWS_MAC_REUSE=0 -DWS_REVMAP=0 -DWS_TWB_INV=0 -DWS_ROT_LATE=0 -DWS_MAC_REGS3=120 -DWS_TMEM_ST=0
FLAGS_r1 := $(R1)
FLAGS_final :=
VARIANTS += wst
FLAGS_wst := -DWS_TIMING=1
SRC_ws2 := pbs_ws2_kernel.cu
FLAGS_ws2 := -DPBS_WS2_NS=ns_ws2 -DPBS_WS2_LAUNCH_NAME=launch_ws2
VARIANTS += ws2t
SRC_ws2t := pbs_ws2_kernel.cu
FLAGS_ws2t := -DPBS_WS2_NS=ns_ws2t -DPBS_WS2_LAUNCH_NAME=launch_ws2t -DWS2_TIMING=1
VARIANTS += ws2w
SRC_ws2w := pbs_ws2_kernel.cu
FLAGS_ws2w := -DPBS_WS2_NS=ns_ws2w -DPBS_WS2_LAUNCH_NAME=launch_ws2w -DWS2_ORDER=0x5761234
