# oracle/metrics.mk -- the checkers of the pose-accuracy metrics (make -f oracle/metrics.mk <target>):
#
#   make -f oracle/metrics.mk nn_oracle -> oracle/libpvnet_nn_oracle.so  (nn_oracle.c: C restatement, OpenMP)
#   make -f oracle/metrics.mk refnn     -> oracle/_ref/libpvnet_refnn.so (the reference's nearest_neighborhood.cu,
#                                          compiled verbatim from where it lies, when it is present)
#
# Both outputs are git-ignored (*.so, oracle/_ref/) but travel to the GPU box.  Same C flags as the voting
# oracle (oracle/Makefile): -march=x86-64-v3 so the .so also runs on the GPU box's host CPU, -ffp-contract=off
# so the FMA placement is the one written in the source.

CC      := gcc
NVCC    ?= nvcc
NN_SRC  ?= /root/reference/lib/utils/extend_utils/src
HERE    := $(dir $(abspath $(lastword $(MAKEFILE_LIST))))

CFLAGS  := -O3 -march=x86-64-v3 -ffp-contract=off -fno-fast-math -fopenmp -fPIC -shared \
           -fvisibility=hidden -Wall -Wextra -std=c11

all: nn_oracle refnn

nn_oracle: $(HERE)libpvnet_nn_oracle.so

$(HERE)libpvnet_nn_oracle.so: $(HERE)nn_oracle.c
	$(CC) $(CFLAGS) -o $@ $< -lm

# nearest_neighborhood.cu is plain CUDA whose extern "C" findNearestPointIdxLauncher takes host pointers:
# compiled verbatim, nothing else is linked in.
refnn:
	@if [ -f $(NN_SRC)/nearest_neighborhood.cu ]; then \
	  mkdir -p $(HERE)_ref && \
	  $(NVCC) -O3 -gencode arch=compute_100a,code=sm_100a -Xcompiler -fPIC -shared \
	    -o $(HERE)_ref/libpvnet_refnn.so $(NN_SRC)/nearest_neighborhood.cu && \
	  echo "built oracle/_ref/libpvnet_refnn.so"; \
	else \
	  echo "reference sources not present at $(NN_SRC); keeping prebuilt oracle/_ref if any"; \
	fi

.PHONY: all nn_oracle refnn
