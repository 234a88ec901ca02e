// Threaded freeimpala harness on the B200 learner path: the reference's cmd/freeimpala/main.cpp wiring
// (setupLearner :175-200, setupAgents :203-231, cleanup :234-260) with the same flags, on top of
// fi_host.hpp. Actor threads stand in for Agent::run (agent.h:230-295): per iteration they produce one
// synthetic trajectory per player in the record layout of DESIGN.md, write it into that player's ring
// (agent.h:96) and then refresh their model copy when a newer version is published (agent.h:155-165).
// BASELINE.json configs[2]: --players 2 --buffer-capacity 32 --batch-size 32 --agents 64.
// Prints one JSON line: learner updates, updates/s, transitions/s (= updates * M * S / wall).
// --sample-actions: on-policy records through the library's own inference. The learner masks illegal actions, and for each
// trajectory an actor draws a random non-empty legal word per record, makes one fi_learner_infer_sample call on the S
// observations, and stores the returned logits (words 162..177), action (178) and legal word (182). The JSON line then also
// reports the rows sampled and how many returned actions fell outside their legal word (always 0).
// --variable-length: games of varying length. The learner trains on each trajectory's own length (variable_length), and an
// actor draws L uniform in 1..game_steps per trajectory, makes and writes only L records (the slot keeps the tail of whatever
// trajectory used it before), with L in word 183 of record 0 and the bootstrap value in record L - 1; with --sample-actions
// it samples those L rows. The JSON line then also reports valid_transitions, the sum of the lengths written.
// --popart-beta B: the learner normalises its value head with PopArt (fi_learner_config.popart_beta); the JSON line then also
// reports each player's final statistics, popart_mu and popart_sigma.
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>

#include "fi_host.hpp"

using namespace fi_host;

struct Params {  // ProgramParams, cmd/freeimpala/main.cpp:18-35 (defaults :38-120)
    size_t players = 2, iterations = 100, entry_size = 100, buffer_capacity = 10, batch_size = 5, learner_time = 500,
           checkpoint_freq = 10, agents = 4, game_steps = 100, agent_time = 200;
    std::string checkpoint_location = "", starting_model = "";
    unsigned seed = 0;
    int infer_every = 0;  // >0: every k-th iteration an actor asks for batched policy inference on its observations
    bool sample_actions = false;
    bool variable_length = false;
    double popart_beta = 0.0;  // --popart-beta B: PopArt value normalisation of the learner (0 = off)
};

static bool parse(int argc, char** argv, Params& p) {
    std::map<std::string, size_t*> num = {{"-p", &p.players}, {"--players", &p.players}, {"-T", &p.iterations},
        {"--iterations", &p.iterations}, {"-S", &p.entry_size}, {"--entry-size", &p.entry_size}, {"-B", &p.buffer_capacity},
        {"--buffer-capacity", &p.buffer_capacity}, {"-M", &p.batch_size}, {"--batch-size", &p.batch_size},
        {"--learner-time", &p.learner_time}, {"-c", &p.checkpoint_freq}, {"--checkpoint-freq", &p.checkpoint_freq},
        {"-a", &p.agents}, {"--agents", &p.agents}, {"--game-steps", &p.game_steps}, {"--agent-time", &p.agent_time}};
    for (int i = 1; i < argc; i++) {
        std::string a = argv[i];
        if (a == "--sample-actions") { p.sample_actions = true; continue; }
        if (a == "--variable-length") { p.variable_length = true; continue; }
        if (i + 1 >= argc) return false;
        if (num.count(a)) *num[a] = strtoull(argv[++i], nullptr, 10);
        else if (a == "-l" || a == "--checkpoint-location") p.checkpoint_location = argv[++i];
        else if (a == "-m" || a == "--starting-model") p.starting_model = argv[++i];
        else if (a == "--seed") p.seed = (unsigned)strtoul(argv[++i], nullptr, 10);
        else if (a == "--infer-every") p.infer_every = atoi(argv[++i]);
        else if (a == "--popart-beta") p.popart_beta = strtod(argv[++i], nullptr);
        else if (a == "--metrics-file" || a == "--log-level" || a == "--broker") ++i;  // accepted, unused here
        else return false;
    }
    // validateParameters, main.cpp:160-172
    if (p.batch_size > p.buffer_capacity) { fprintf(stderr, "Batch size (M) must be <= buffer capacity (B)\n"); return false; }
    if (p.game_steps > p.entry_size) { fprintf(stderr, "Game steps must be <= entry size (S)\n"); return false; }
    if (p.variable_length && p.game_steps == 0) { fprintf(stderr, "--variable-length needs game steps >= 1\n"); return false; }
    return true;
}

struct SampleCounts {
    std::atomic<uint64_t> rows{0}, illegal{0}, valid_transitions{0};
    std::atomic<bool> failed{false};
};

static void actor(size_t id, const Params& P, Learner& learner, std::atomic<uint64_t>& inferences, SampleCounts& sampled) {
    auto buffers = learner.getSharedBuffers();
    auto models = learner.getModelManager();
    std::vector<uint64_t> versions(P.players, 0);
    std::vector<std::shared_ptr<Model>> local(P.players);
    for (size_t p = 0; p < P.players; p++) {
        local[p] = models->getModel(p);
        versions[p] = local[p] ? local[p]->getVersion() : 0;
    }
    std::vector<float> slot(P.entry_size * 256, 0.f);
    uint64_t rng = 0x9E3779B97F4A7C15ull * (id + 1) + P.seed;
    auto next = [&] { rng ^= rng << 13; rng ^= rng >> 7; rng ^= rng << 17; return rng; };
    auto unif = [&] { return (float)((next() >> 40) * (1.0 / 16777216.0)) * 2.f - 1.f; };
    for (size_t it = 0; it < P.iterations; it++) {
        if (P.agent_time) std::this_thread::sleep_for(std::chrono::milliseconds(P.agent_time));  // agent.h:41
        for (size_t p = 0; p < P.players; p++) {
            // the game's length: entry_size records, or (--variable-length) L uniform in 1..game_steps
            const size_t len = P.variable_length ? 1 + next() % P.game_steps : P.entry_size;
            // simulateGame (agent.h:34-75): game_steps records, here with a well-formed transition in each
            for (size_t s = 0; s < len; s++) {
                float* rec = slot.data() + s * 256;
                for (int j = 0; j < 178; j++) rec[j] = unif();           // observation + behaviour logits
                int32_t act = (int32_t)(next() % 16);
                memcpy(rec + 178, &act, 4);
                rec[179] = unif();                                       // reward
                rec[180] = (next() % 100) ? 0.99f : 0.f;                 // discount = 0.99 (1 - done)
                rec[181] = s + 1 == len ? unif() : 0.f;                  // bootstrap value in the last record
            }
            if (P.variable_length) {
                const uint32_t w = (uint32_t)len;
                memcpy(slot.data() + FI_REC_WORD_LENGTH, &w, 4);         // the length, in record 0
                sampled.valid_transitions.fetch_add(len);
            }
            if (P.sample_actions) {   // the policy's own logits and actions over a random legal set per record
                std::vector<float> obs(len * 162), logits(len * 16);
                std::vector<uint32_t> legal(len);
                std::vector<int32_t> acts(len);
                for (size_t s = 0; s < len; s++) {
                    memcpy(&obs[s * 162], &slot[s * 256], 162 * 4);
                    do legal[s] = (uint32_t)(next() & 0xFFFF); while (legal[s] == 0);
                }
                const uint64_t seed = ((uint64_t)id << 40) ^ ((uint64_t)it << 8) ^ p;
                if (fi_learner_infer_sample(learner.handle(), (int)p, obs.data(), legal.data(), len, seed, 0, acts.data(),
                                            logits.data(), nullptr) != FI_OK) {
                    fprintf(stderr, "freeimpala_gpu: fi_learner_infer_sample: %s\n", fi_last_error());
                    sampled.failed.store(true);
                } else {
                    sampled.rows.fetch_add(len);
                    for (size_t s = 0; s < len; s++) {
                        float* rec = slot.data() + s * 256;
                        if (acts[s] < 0 || acts[s] >= 16 || !((legal[s] >> acts[s]) & 1u)) sampled.illegal.fetch_add(1);
                        memcpy(rec + 162, &logits[s * 16], 16 * 4);
                        memcpy(rec + 178, &acts[s], 4);
                        memcpy(rec + FI_REC_WORD_LEGAL, &legal[s], 4);
                    }
                }
            }
            if (P.infer_every && it % P.infer_every == 0) {              // batched actor policy inference
                std::vector<float> obs(P.entry_size * 162), logits(P.entry_size * 16), values(P.entry_size);
                for (size_t s = 0; s < P.entry_size; s++) memcpy(&obs[s * 162], &slot[s * 256], 162 * 4);
                if (fi_learner_infer(learner.handle(), (int)p, obs.data(), nullptr, P.entry_size, 0, logits.data(), values.data()) == FI_OK)
                    inferences.fetch_add(P.entry_size);
            }
            buffers[p]->write(slot.data(), len * 256 * sizeof(float));     // transferThread, agent.h:96
        }
        for (size_t p = 0; p < P.players; p++) {                          // modelUpdateThread, agent.h:155-165
            const uint64_t latest = models->getLatestVersion(p);
            if (latest > versions[p]) {
                local[p] = models->getModel(p);
                if (local[p]) versions[p] = local[p]->getVersion();
            }
        }
    }
}

int main(int argc, char** argv) {
    Params P;
    if (!parse(argc, argv, P)) {
        fprintf(stderr, "usage: freeimpala_gpu [-p N] [-T N] [-S N] [-B N] [-M N] [-a N] [--game-steps N] [--agent-time ms] "
                        "[-c N] [-l DIR] [-m DIR] [--seed N] [--infer-every K] [--sample-actions] [--variable-length] [--popart-beta B]\n");
        return 2;
    }
    const size_t learner_iterations = (P.agents * P.iterations) / P.batch_size;  // main.cpp:179 (integer division)
    try {
        Learner learner(P.players, P.buffer_capacity, P.entry_size, P.batch_size, P.learner_time, P.checkpoint_freq,
                        P.checkpoint_location, P.starting_model, learner_iterations, 0, FI_MODEL_MLP_ACTOR_CRITIC,
                        P.sample_actions, P.variable_length, false, P.popart_beta);
        const auto t0 = std::chrono::steady_clock::now();
        learner.start();
        std::atomic<uint64_t> inferences{0};
        SampleCounts sampled;
        std::vector<std::thread> threads;
        for (size_t a = 0; a < P.agents; a++) threads.emplace_back([&, a] { actor(a, P, learner, inferences, sampled); });
        for (auto& t : threads) t.join();
        // The reference stops the learner as soon as the agents have joined (main.cpp:239-246), which drops whatever
        // the workers have not consumed yet. Every trajectory needed for learner_iterations updates has been written
        // at this point, so let the workers finish them (bounded wait) to make the run deterministic.
        const auto deadline = std::chrono::steady_clock::now() + std::chrono::seconds(120);
        auto done = [&] { size_t u = 0; for (size_t p = 0; p < P.players; p++) u += learner.iterationsDone(p); return u; };
        while (done() < learner_iterations * P.players && !learner.failed() && std::chrono::steady_clock::now() < deadline)
            std::this_thread::sleep_for(std::chrono::microseconds(200));
        learner.stop();
        const double sec = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        size_t updates = 0;
        for (size_t p = 0; p < P.players; p++) updates += learner.iterationsDone(p);
        uint64_t inf_calls = 0, inf_batches = 0;   // concurrent actors' requests are combined into few forwards per player
        for (size_t p = 0; p < P.players; p++) {
            uint64_t c = 0, b = 0;
            fi_learner_infer_stats(learner.handle(), (int)p, &c, &b, nullptr);
            inf_calls += c;
            inf_batches += b;
        }
        uint64_t vmin = ~0ull;
        for (size_t p = 0; p < P.players; p++) vmin = std::min<uint64_t>(vmin, learner.getModelManager()->getLatestVersion(p));
        printf("{\"harness\": \"freeimpala_gpu\", \"players\": %zu, \"agents\": %zu, \"batch_size\": %zu, \"entry_size\": %zu, "
               "\"learner_updates\": %zu, \"expected_updates\": %zu, \"seconds\": %.4f, \"updates_per_s\": %.2f, "
               "\"transitions_per_s\": %.1f, \"min_model_version\": %llu, \"actor_inference_rows\": %llu, "
               "\"actor_inference_calls\": %llu, \"actor_inference_forwards\": %llu, \"kernel_launches\": %llu",
               P.players, P.agents, P.batch_size, P.entry_size, updates, learner_iterations * P.players, sec, updates / sec,
               updates * (double)P.batch_size * P.entry_size / sec, (unsigned long long)vmin,
               (unsigned long long)inferences.load(), (unsigned long long)inf_calls, (unsigned long long)inf_batches,
               (unsigned long long)fi_kernel_launch_count());
        if (P.sample_actions)
            printf(", \"actor_sampled_rows\": %llu, \"illegal_actions\": %llu", (unsigned long long)sampled.rows.load(),
                   (unsigned long long)sampled.illegal.load());
        if (P.variable_length) printf(", \"valid_transitions\": %llu", (unsigned long long)sampled.valid_transitions.load());
        if (P.popart_beta > 0.0) {   // each player's final PopArt statistics
            std::string mus, sigmas;
            for (size_t p = 0; p < P.players; p++) {
                double st[3] = {0.0, 0.0, 0.0};
                if (fi_learner_popart_stats(learner.handle(), (int)p, st) != FI_OK) {
                    fprintf(stderr, "freeimpala_gpu: fi_learner_popart_stats: %s\n", fi_last_error());
                    return 1;
                }
                char buf[64];
                snprintf(buf, sizeof(buf), "%s%.17g", p ? ", " : "", st[0]);
                mus += buf;
                snprintf(buf, sizeof(buf), "%s%.17g", p ? ", " : "", st[2]);
                sigmas += buf;
            }
            printf(", \"popart_mu\": [%s], \"popart_sigma\": [%s]", mus.c_str(), sigmas.c_str());
        }
        printf("}\n");
        if (sampled.failed.load() || sampled.illegal.load()) return 1;
        return updates == learner_iterations * P.players ? 0 : 1;
    } catch (const std::exception& e) {
        fprintf(stderr, "freeimpala_gpu: %s\n", e.what());
        return 3;
    }
}
