# Builds the product library (CUDA, sm_100a), the peaks microbenchmark and the test oracle.
NVCC      ?= /usr/local/cuda/bin/nvcc
ARCH      := -gencode arch=compute_100a,code=sm_100a
NVCCFLAGS := $(ARCH) -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xptxas -v
CSRC      := bisip_b200/csrc
LIB       := $(CSRC)/libbisip_b200.so
HDRS      := $(wildcard $(CSRC)/*.cuh) include/bisip_b200.h

all: $(LIB) tools/peaks oracle

# One object per kernel family so that they compile in parallel (`make -j`); no device code crosses a
# translation unit, so a plain host link is enough.  ptxas -v output of every unit is kept in $(CSRC)/ptxas.log.
UNITS     := api ens_wp_collapsed ens_wp_vec ens_wp_dmma ens_dmma ens_rc ens_umma ens_collapsed ens_colecole ens_dias_shin batch_decomp batch_vec
OBJS      := $(UNITS:%=$(CSRC)/%.o)

$(CSRC)/%.o: $(CSRC)/%.cu $(HDRS)
	$(NVCC) $(NVCCFLAGS) -c -o $@ $< 2> $(CSRC)/$*.ptxas || (cat $(CSRC)/$*.ptxas; false)

$(LIB): $(OBJS)
	$(NVCC) $(ARCH) -shared -o $@ $(OBJS)
	cat $(UNITS:%=$(CSRC)/%.ptxas) > $(CSRC)/ptxas.log

# developer build with per-phase cycle counters (not shipped, not loaded by the package)
dbg: $(HDRS)
	$(NVCC) $(ARCH) -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -shared -DBISIP_PHASE_TIMING -o $(CSRC)/libbisip_b200_dbg.so $(UNITS:%=$(CSRC)/%.cu)

tools/peaks: tools/peaks.cu
	$(NVCC) $(ARCH) -O3 -lineinfo -o $@ $<

oracle:
	python -c "from oracle import oracle; oracle.build()"
	./oracle/build_ref.sh

clean:
	rm -f $(LIB) $(OBJS) $(CSRC)/*.ptxas tools/peaks $(CSRC)/ptxas.log
	rm -rf oracle/_build

.PHONY: all oracle clean dbg
