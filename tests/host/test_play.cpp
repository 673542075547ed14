// Standalone test of alphazero_risk_b200/host/az_play.hpp with a mirror of the reference's GameResults (game/game.h:10-29).
// Without a GPU: construction must fail loudly -> NO_DEVICE_OK.  With a GPU: a 40-game match (--mcts=16, -t 2) -> PLAY_OK.
// Usage: test_play [DIR]; with a GPU, DIR (required) receives the checkpoint the test writes.
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>
#include "az_play.hpp"

struct PlayerGameResult { int win = 0; int winAndStartedGame = 0; };
struct GameResults { int count = 0; int draw = 0; std::vector<PlayerGameResult> players = std::vector<PlayerGameResult>(2); };

int main(int argc, char** argv)
{
    azb200::PlaySettings s;
    s.MCTS_SIMULATIONS = 16; s.THREADS_PER_MCTS = 2; s.BLOCKS = 2;
    if (az_device_count() == 0) {
        try { azb200::DevicePlay p(s); }
        catch (const std::runtime_error& e) { printf("NO_DEVICE_OK %s\n", e.what()); return 0; }
        printf("expected a failure without a GPU\n");
        return 1;
    }
    if (argc < 2) { printf("usage: %s DIR (the checkpoint the test writes goes there)\n", argv[0]); return 2; }
    const std::string ck = std::string(argv[1]) + "/az_b200_play_ckpt";
    azb200::DevicePlay p(s);
    remove((ck + ".index").c_str()); remove((ck + ".data-00000-of-00001").c_str());
    p.loadCheckpoint(ck);            // missing: random init kept and saved as a TensorFlow checkpoint bundle
    GameResults a = p.playGames<GameResults>(41);          // odd request: 40 games, like Counter::hasNext(2)
    GameResults b = p.playGames<GameResults>(41);          // same seed, same weights: the match is reproducible
    bool ok = a.count == 40 && a.draw + a.players[0].win + a.players[1].win == 40 &&
              a.players[0].winAndStartedGame <= a.players[0].win && a.players[1].winAndStartedGame <= a.players[1].win &&
              b.count == a.count && b.draw == a.draw && b.players[0].win == a.players[0].win && b.players[1].win == a.players[1].win;
    // the trainer's comparison match: a second DevicePlay holds the "old" model (here the same checkpoint), player index 1 searches
    // with its network and its own tables
    azb200::DevicePlay old(s);
    old.loadCheckpoint(ck);
    p.setOpponentNetwork(old.network());
    GameResults c = p.playGames<GameResults>(12);
    ok = ok && c.count == 12 && c.draw + c.players[0].win + c.players[1].win == 12 && p.last.opponent_turns > 0 && p.last.az_moves > 0;
    p.setOpponent(AZ_OPPONENT_RANDOM);                     // the trainer's benchmark opponent
    GameResults d = p.playGames<GameResults>(6);
    ok = ok && d.count == 6;
    // trainOnGeneratedData's bootstrap games: Script vs Random with every Player::addTrainingSample recorded, then three epochs on them
    {
        azb200::DeviceDataGames gen(s, 24);
        std::vector<uint8_t> recs = gen.play(30, true);        // 30 games asked: two batches of 24
        const size_t nrec = recs.size() / AZ_SAMPLE_BYTES;
        bool data_ok = gen.games_played == 48 && gen.dropped == 0 && nrec > 48 * 100 && recs.size() % AZ_SAMPLE_BYTES == 0;
        for (size_t i = 0; data_ok && i < nrec; i += 97) {     // one-hot policy, value in {-1, 0, 1}, player byte = NNInputData::playerIndex
            const uint8_t* r = recs.data() + i * AZ_SAMPLE_BYTES;
            float v, pol[43]; memcpy(&v, r + 89, 4); memcpy(pol, r + 93, sizeof pol);
            int ones = 0, zeros = 0;
            for (float x : pol) { ones += x == 1.0f; zeros += x == 0.0f; }
            data_ok = ones == 1 && zeros == 42 && (v == 1.0f || v == -1.0f || v == 0.0f) && r[0] < 2 && r[0] == r[1 + 42];
        }
        float lp[3] = { 0, 0, 0 }, lv[3] = { 0, 0, 0 };
        data_ok = data_ok && az_nn_train(p.network(), recs.data(), nrec, 3, 512, 7, lp, lv, nullptr) == AZ_OK && lp[2] < lp[0];
        printf("%s bootstrap games %d samples %zu policy loss %.3f -> %.3f\n", data_ok ? "DATA_OK" : "DATA_FAIL", gen.games_played, nrec, lp[0], lp[2]);
        ok = ok && data_ok;
    }
    printf("%s count=%d draw=%d az=%d/%d script=%d/%d | new vs old %d/%d %d/%d draw %d | vs random az %d of %d\n", ok ? "PLAY_OK" : "PLAY_FAIL",
           a.count, a.draw, a.players[0].win, a.players[0].winAndStartedGame, a.players[1].win, a.players[1].winAndStartedGame,
           c.players[0].win, c.players[0].winAndStartedGame, c.players[1].win, c.players[1].winAndStartedGame, c.draw, d.players[0].win, d.count);
    return ok ? 0 : 1;
}
