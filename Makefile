# Top-level build: the product library + CLI (sm_100a only) and the test-only oracle.
#   make            -> phfpfac_b200/_build/libpfac_b200.so, phfpfac_b200/_build/gphf, oracle
#   make lib | cli | oracle
NVCC ?= /usr/local/cuda/bin/nvcc
HOSTCXX := g++
ARCH := -gencode arch=compute_100a,code=sm_100a
B := phfpfac_b200/_build
SRC := phfpfac_b200/csrc
NVFLAGS := $(EXTRA) $(ARCH) -lineinfo -O3 -std=c++17 -ccbin $(HOSTCXX) -Iinclude -I$(SRC) \
           -Xcompiler -fPIC,-Wall,-Wextra,-pthread -Xptxas -v
HOST_SRCS := $(SRC)/pfac_tables.cc $(SRC)/pfac_writer.cc $(SRC)/pfac_job.cc $(SRC)/pfac_derive.cc
CUDA_SRCS := $(SRC)/pfac_device.cu
HDRS := include/pfac_b200.h $(SRC)/pfac_internal.h $(SRC)/pfac_kernel.cuh $(SRC)/pfac_compact.cuh $(SRC)/pfac_batch.cuh $(SRC)/pfac_flows.cuh $(SRC)/pfac_fold.cuh $(SRC)/pfac_rules.cuh $(SRC)/pfac_derive.h

.PHONY: all lib cli oracle synth clean
all: lib cli oracle synth

# workload generators of the tests and bench.py: a tools library, not part of the product ABI
synth: tools/_build/libpfac_synth.so
tools/_build/libpfac_synth.so: tools/synth/pfac_synth.cc tools/synth/pfac_synth.h
	@mkdir -p tools/_build
	$(HOSTCXX) -O2 -std=c++17 -Wall -Wextra -fPIC -shared -pthread -Itools/synth -o $@ tools/synth/pfac_synth.cc

lib: $(B)/libpfac_b200.so
cli: $(B)/gphf

$(B)/libpfac_b200.so: $(HOST_SRCS) $(CUDA_SRCS) $(HDRS)
	@mkdir -p $(B)
	$(NVCC) $(NVFLAGS) -shared -cudart static -o $@ $(CUDA_SRCS) $(HOST_SRCS) 2> $(B)/ptxas.log || (cat $(B)/ptxas.log; false)
	@grep -E "registers|spill|error" $(B)/ptxas.log | head -20 || true

$(B)/gphf: $(SRC)/gphf_main.cc $(B)/libpfac_b200.so
	$(HOSTCXX) -O2 -std=c++17 -Wall -Wextra -Iinclude -o $@ $(SRC)/gphf_main.cc -L$(B) -lpfac_b200 -Wl,-rpath,'$$ORIGIN'

oracle:
	$(MAKE) -C oracle all

# development: a variant of the library under another name, e.g.
#   make variant NAME=w23 EXTRA=-DPFAC_CONSUMER_WARPS=23   ->  $(B)/libpfac_b200_w23.so  (PFAC_B200_LIB=... selects it)
variant:
	@mkdir -p $(B)
	$(NVCC) $(NVFLAGS) -shared -cudart static -o $(B)/libpfac_b200_$(NAME).so $(CUDA_SRCS) $(HOST_SRCS) 2> $(B)/ptxas_$(NAME).log || (cat $(B)/ptxas_$(NAME).log; false)

clean:
	rm -rf $(B) tools/_build
	$(MAKE) -C oracle clean
