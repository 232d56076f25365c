# Builds libgpud_b200.so (sm_100a only) and the oracle.  `python -c "import __graft_entry__ as g; g.build()"` calls this.
NVCC ?= /usr/local/cuda/bin/nvcc
ARCH := -gencode arch=compute_100a,code=sm_100a
NVFLAGS := $(ARCH) -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xcompiler -Wall -Xptxas -v $(if $(EXPERIMENT_TMA),-DGPUD_EXPERIMENT_TMA)
SRC := gpud_b200/csrc
OBJS := $(SRC)/api.o $(SRC)/ring.o $(SRC)/select.o $(SRC)/kmsg_scan.o $(SRC)/ib_scan.o $(SRC)/fabric.o $(SRC)/catalog.o $(SRC)/host_component.o $(SRC)/component_abi.o $(SRC)/kmsg_stateful.o $(SRC)/poller.o $(SRC)/store_sqlite.o
LIB := gpud_b200/libgpud_b200.so

all: $(LIB) gpud_b200/gpud-scan oracle

$(SRC)/%.o: $(SRC)/%.cu $(SRC)/internal.h $(SRC)/catalog.h $(SRC)/ring_drain.h include/gpud_b200.h
	$(NVCC) $(NVFLAGS) -c $< -o $@ 2> $@.ptxas.log || (cat $@.ptxas.log; exit 1)

$(SRC)/catalog.o: $(SRC)/catalog.cpp $(SRC)/catalog.h $(SRC)/catalog_data.inc include/gpud_b200.h
	g++ -O2 -std=c++17 -fPIC -Wall -c $< -o $@

$(SRC)/host_component.o: $(SRC)/host_component.cpp $(SRC)/host_component.h $(SRC)/json_min.h include/gpud_b200.h
	g++ -O2 -std=c++17 -fPIC -Wall -c $< -o $@

$(SRC)/component_abi.o: $(SRC)/component_abi.cpp $(SRC)/host_component.h $(SRC)/internal.h $(SRC)/ring_drain.h include/gpud_b200.h
	g++ -O2 -std=c++17 -fPIC -Wall -I/usr/local/cuda/include -c $< -o $@

$(SRC)/poller.o: $(SRC)/poller.cpp $(SRC)/internal.h include/gpud_b200.h
	g++ -O2 -std=c++17 -fPIC -Wall -I/usr/local/cuda/include -c $< -o $@

$(SRC)/store_sqlite.o: $(SRC)/store_sqlite.cpp $(SRC)/json_min.h $(SRC)/ring_drain.h include/gpud_b200.h
	g++ -O2 -std=c++17 -fPIC -Wall -c $< -o $@

$(SRC)/kmsg_stateful.o: $(SRC)/kmsg_stateful.cpp include/gpud_b200.h
	g++ -O2 -std=c++17 -fPIC -Wall -c $< -o $@

# BASELINE configs[0]: the `gpud scan`-shaped one-shot for a CPU-only host; no CUDA, no library
gpud_b200/gpud-scan: $(SRC)/scan_main.cpp
	g++ -O2 -std=c++17 -Wall -o $@ $<

$(LIB): $(OBJS)
	$(NVCC) $(ARCH) -shared -o $@ $(OBJS) -lcudart -ldl

oracle:
	$(MAKE) -C oracle

clean:
	rm -f $(SRC)/*.o $(SRC)/*.ptxas.log $(LIB) gpud_b200/gpud-scan
	$(MAKE) -C oracle clean

.PHONY: all oracle clean
