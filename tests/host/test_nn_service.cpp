// Standalone test of the host adapter (alphazero_risk_b200/host/az_nn_service.hpp) with the mirror types.
// Without a GPU: constructing the service must fail loudly (no CPU fallback) -> prints NO_DEVICE_OK.
// With a GPU: 16 threads call registerThread / predictFuture concurrently like the reference's search threads;
// every future must equal a direct az_nn_forward of the same input -> prints SERVICE_OK <batches>.
// Usage: test_nn_service [DIR]; with a GPU, DIR (required) receives the checkpoints the test writes.
#include <atomic>
#include <cmath>
#include <cstdio>
#include <filesystem>
#include <thread>
#include "az_nn_service.hpp"

using namespace azb200;
typedef AlphaZeroClusterT<NNInputData, NNOutputData, NNTrainData> Cluster;

static NNInputData make_input(unsigned k)
{
    NNInputData in;
    for (int i = 0; i < 42; ++i) { in.land[i].army = 1 + (k * 7 + i * 3) % 30; in.land[i].playerIndex = (k + i) % 3; }
    in.playerIndex = k & 1; in.round = 1 + k % 50;
    in.featureReinforcementShare = 0.25f + 0.01f * (k % 40); in.featureAttackFrequency = 0.125f * (k % 9); in.featureCanDrawCard = k % 2;
    in.featureIsPhaseAttack = 1.0f; in.featureArmyShare = 0.3f + 0.005f * (k % 60);
    return in;
}

int main(int argc, char** argv)
{
    static_assert(sizeof(NNInputData) == 88, "mirror layout");
    if (az_device_count() == 0) {
        try { Cluster c(AZ_NN_FP32, 2); c.initGpus(1); c.initPlayerGroup("az1", "model_bin_V2_2.pb"); }
        catch (const std::runtime_error& e) { printf("NO_DEVICE_OK %s\n", e.what()); return 0; }
        printf("expected a failure without a GPU\n");
        return 1;
    }
    Cluster cluster(AZ_NN_FP32, 2);
    cluster.initGpus(1);
    auto group = cluster.initPlayerGroup("az1", "model_bin_V2_2.pb");
    bool dup = false;
    try { cluster.initPlayerGroup("az1", "model_bin_V2_2.pb"); } catch (const std::invalid_argument&) { dup = true; }   // upstream behaviour
    if (!dup) { printf("duplicate group accepted\n"); return 1; }
    if (argc < 2) { printf("usage: %s DIR (the checkpoints the test writes go there)\n", argv[0]); return 2; }
    const std::string ck = std::string(argv[1]) + "/az_b200_test_ckpt";
    auto nn = group->getNN(0);
    std::filesystem::remove_all(ck);
    nn->loadCheckpoint(ck + "/az1");          // missing -> random init + save (a TensorFlow checkpoint bundle)
    if (!std::filesystem::exists(ck + "/az1.index") || !std::filesystem::exists(ck + "/az1.data-00000-of-00001")) {
        printf("checkpoint bundle was not written\n"); return 1; }
    const int T = 16, R = 40;
    std::atomic<int> bad{ 0 };
    std::vector<std::thread> th;
    for (int t = 0; t < T; ++t)
        th.emplace_back([&, t]() {
            nn->registerThread();
            for (int r = 0; r < R; ++r) {
                NNInputData in = make_input(t * 1000 + r);
                NNOutputData a = nn->predictFuture(in).get();
                NNOutputData b = nn->predict(in);
                if (a.policy.size() != 43 || b.policy.size() != 43 || a.value != b.value) { bad++; continue; }
                float s = 0;
                for (int i = 0; i < 43; ++i) { if (a.policy[i] != b.policy[i]) bad++; s += a.policy[i]; }
                if (std::fabs(s - 1.0f) > 1e-4f) bad++;
            }
            nn->unregisterThread();
        });
    for (auto& x : th) x.join();
    // AlphaZeroNNGroup::train (alphazero_nn.cpp:351-410): 2 epochs over 96 samples in batches of 32 must change the predictions,
    // and a checkpoint written afterwards must restore them in a second group
    std::vector<NNTrainData> data;
    for (unsigned k = 0; k < 96; ++k) {
        NNTrainData td; td.playerIndex = (int8_t)(k & 1); td.in = make_input(5000 + k);
        td.out.policy.assign(43, 0.0f); td.out.policy[k % 43] = 0.75f; td.out.policy[(k * 5 + 1) % 43] += 0.25f;
        td.out.value = (k % 3 == 0) ? 1.0f : -1.0f;
        data.push_back(td);
    }
    NNInputData probe = make_input(777);
    NNOutputData before = nn->predict(probe);
    nn->service().setBatchSize(32);
    group->train(data, 2);
    NNOutputData after = nn->predict(probe);
    bool moved = before.value != after.value;
    group->saveCheckpoint(ck + "/trained");
    auto group2 = cluster.initPlayerGroup("az2", "model_bin_V2_2.pb");
    group2->loadCheckpoint(ck + "/trained");
    NNOutputData again = group2->getNN(0)->predict(probe);
    bool restored = again.value == after.value;
    for (int i = 0; i < 43; ++i) restored = restored && again.policy[i] == after.policy[i];
    // the group hand-off after train (alphazero_gpu_cluster.cpp:221-231) without the temporary checkpoint file: a third network takes
    // the trained state device to device; with >= 2 GPUs the group itself spans two devices and train() must leave both copies equal
    auto group3 = cluster.initPlayerGroup("az3", "model_bin_V2_2.pb");
    group3->getNN(0)->service().initRandom(99);
    group3->getNN(0)->service().copyStateFrom(nn->service());
    NNOutputData copied = group3->getNN(0)->predict(probe);
    for (int i = 0; i < 43; ++i) restored = restored && copied.policy[i] == after.policy[i];
    restored = restored && copied.value == after.value;
    if (az_device_count() >= 2) {
        Cluster two(AZ_NN_FP32, 2);
        two.initGpus(2);
        auto g2 = two.initPlayerGroup("pair", "model_bin_V2_2.pb");
        g2->loadCheckpoint(ck + "/az1");
        g2->getNN(0)->service().setBatchSize(32);
        g2->train(data, 1);
        NNOutputData p0 = g2->getNN(0)->predict(probe), p1 = g2->getNN(1)->predict(probe);
        for (int i = 0; i < 43; ++i) restored = restored && p0.policy[i] == p1.policy[i];
        restored = restored && p0.value == p1.value && p0.value != before.value;
        printf("two-GPU group hand-off checked\n");
    }
    if (bad || !moved || !restored) { printf("SERVICE_FAIL bad=%d moved=%d restored=%d\n", bad.load(), (int)moved, (int)restored); return 1; }
    printf("SERVICE_OK\n");
    return 0;
}
