# Builds libcopra_b200.so (C ABI + sm_100a kernels) in-tree, and the CPU oracle (test infrastructure).
NVCC ?= nvcc
ARCH := -gencode arch=compute_100a,code=sm_100a
EXTRA ?=
NVFLAGS := $(ARCH) -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xptxas -v $(EXTRA)
CSRC := copra_b200/csrc
OBJS := $(CSRC)/k6_solver.o $(CSRC)/k6_thin.o $(CSRC)/k6_thin_f0.o $(CSRC)/k6_thin_f1.o $(CSRC)/k6_thin_f2.o $(CSRC)/k6_thin_cluster.o $(CSRC)/k1_k7_lmpc.o $(CSRC)/dgemm_dmma.o $(CSRC)/fp64_peak.o $(CSRC)/k8_k9_sens.o $(CSRC)/capi.o $(CSRC)/capi_multi.o
LIB := copra_b200/lib/libcopra_b200.so
HDRS := $(wildcard $(CSRC)/*.cuh) $(wildcard $(CSRC)/*.h) include/copra_b200.h

all: $(LIB) oracle tests/cpp/test_facade tests/cpp/test_per_step tests/cpp/test_vjp tests/cpp/test_jvp tests/cpp/test_vjp_costs tests/cpp/test_vjp_model tests/cpp/test_initial_state_sens

$(CSRC)/%.o: $(CSRC)/%.cu $(HDRS)
	$(NVCC) $(NVFLAGS) -c $< -o $@ 2> $@.ptxas.log || (cat $@.ptxas.log; false)

$(LIB): $(OBJS)
	mkdir -p copra_b200/lib
	$(NVCC) $(ARCH) -shared -o $@ $(OBJS) -cudart static -ldl

oracle:
	$(MAKE) -C oracle -s

clean:
	rm -f $(OBJS) $(CSRC)/*.ptxas.log $(LIB)
	$(MAKE) -C oracle clean

.PHONY: all oracle clean

# C++ facade tests (reference test scenarios against include/copra/*)
tests/cpp/test_facade: tests/cpp/test_facade.cpp tests/cpp/systems.hpp $(wildcard include/copra/*) include/copra_b200.h $(LIB)
	g++ -std=c++14 -O1 -Wall -Wextra -pthread -Iinclude -o $@ tests/cpp/test_facade.cpp -Lcopra_b200/lib -lcopra_b200 -Wl,-rpath,'$$ORIGIN/../../copra_b200/lib'

facade-test: tests/cpp/test_facade

# BatchedLMPC with per-step references and limits + retarget (needs the GPU to run)
tests/cpp/test_per_step: tests/cpp/test_per_step.cpp $(wildcard include/copra/*) include/copra_b200.h $(LIB)
	g++ -std=c++14 -O1 -Wall -Wextra -pthread -Iinclude -o $@ tests/cpp/test_per_step.cpp -Lcopra_b200/lib -lcopra_b200 -Wl,-rpath,'$$ORIGIN/../../copra_b200/lib'

per-step-test: tests/cpp/test_per_step

# BatchedLMPC::vjp against central differences of per-instance copra::LMPC solves, and its errors (needs the GPU to run)
tests/cpp/test_vjp: tests/cpp/test_vjp.cpp $(wildcard include/copra/*) include/copra_b200.h $(LIB)
	g++ -std=c++14 -O1 -Wall -Wextra -pthread -Iinclude -o $@ tests/cpp/test_vjp.cpp -Lcopra_b200/lib -lcopra_b200 -Wl,-rpath,'$$ORIGIN/../../copra_b200/lib'

vjp-test: tests/cpp/test_vjp

# BatchedLMPC::feedbackGain / ::jvp against central differences of per-instance copra::LMPC solves, and their errors (GPU)
tests/cpp/test_jvp: tests/cpp/test_jvp.cpp $(wildcard include/copra/*) include/copra_b200.h $(LIB)
	g++ -std=c++14 -O1 -Wall -Wextra -pthread -Iinclude -o $@ tests/cpp/test_jvp.cpp -Lcopra_b200/lib -lcopra_b200 -Wl,-rpath,'$$ORIGIN/../../copra_b200/lib'

jvp-test: tests/cpp/test_jvp

# BatchedLMPC::vjp with the cost gradients: writes them for tests/test_vjp_costs_gpu.py, checks its errors (GPU)
tests/cpp/test_vjp_costs: tests/cpp/test_vjp_costs.cpp $(wildcard include/copra/*) include/copra_b200.h $(LIB)
	g++ -std=c++14 -O1 -Wall -Wextra -pthread -Iinclude -o $@ tests/cpp/test_vjp_costs.cpp -Lcopra_b200/lib -lcopra_b200 -Wl,-rpath,'$$ORIGIN/../../copra_b200/lib'

vjp-costs-test: tests/cpp/test_vjp_costs

# BatchedLMPC::vjp with the model gradients against central differences of copra::LMPC, and its errors (GPU)
tests/cpp/test_vjp_model: tests/cpp/test_vjp_model.cpp $(wildcard include/copra/*) include/copra_b200.h $(LIB)
	g++ -std=c++14 -O1 -Wall -Wextra -pthread -Iinclude -o $@ tests/cpp/test_vjp_model.cpp -Lcopra_b200/lib -lcopra_b200 -Wl,-rpath,'$$ORIGIN/../../copra_b200/lib'

vjp-model-test: tests/cpp/test_vjp_model

# BatchedLMPC::initialStateVjp / initialStateJvp on an initial-state controller (needs the GPU to run)
tests/cpp/test_initial_state_sens: tests/cpp/test_initial_state_sens.cpp $(wildcard include/copra/*) include/copra_b200.h $(LIB)
	g++ -std=c++14 -O1 -Wall -Wextra -pthread -Iinclude -o $@ tests/cpp/test_initial_state_sens.cpp -Lcopra_b200/lib -lcopra_b200 -Wl,-rpath,'$$ORIGIN/../../copra_b200/lib'

initial-state-sens-test: tests/cpp/test_initial_state_sens
